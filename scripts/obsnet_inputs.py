"""What building ObsNet's training inputs in one call saves over stitching the separate calls together (GPU).

    python scripts/obsnet_inputs.py [--rounds R] [--steps K] [--batch B] [--json FILE]

Inputs: B = 20 samples (the shipped ObsNet batch); B synthetic 2000 x 1000 envmaps held in an ``EnvmapBank``, rendered
through a permutation of its slots; zK ~ U[0,1]^6 and equatorial views; B sphere normal maps of 512 x 512
(synth.sphere_normals(256), normalise(n + N(0, 0.05)) inside the sphere, channel-first) with ObsNet's mask
||n|| > 0.5; res 128, thr pi/256, the renderer's footprint chosen on the device.

Each step goes from those device tensors to ObsNet's inputs (cond, mask, transformed LrK, parameters, raw refmap and
mask):
  (a) hand-stitched: render_batch, then per image boolean-mask compaction of the normals, refmap_lookup and
      refmap_mask_make, then obsnet_condition and normalized_log_apply;
  (b) obsnet_inputs.
Per step: device time between CUDA events around the step, and host wall time with a final synchronise.  (a), (b) and
the render alone alternate R times in one process after a warm-up; the outputs of (a) and (b) are checked equal in the
same run, and the card's name and power limit are read in the same run.
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
    ap.add_argument("--batch", type=int, default=20)
    ap.add_argument("--json", default=str(ROOT / "profiles" / "r9_obsnet_inputs.json"))
    args = ap.parse_args()
    if args.rounds < 3 or args.steps < 1 or args.batch < 1:
        ap.error("--rounds >= 3, --steps >= 1, --batch >= 1")

    import numpy as np
    import torch

    from drmnet_b200.callers import (normalized_log_apply, obsnet_condition, obsnet_inputs, refmap_lookup)
    from drmnet_b200.img2refmap import refmap_mask_make
    from drmnet_b200.renderer import B200RefMapRenderer, EnvmapBank, render_batch
    from drmnet_b200.synth import BRDF_PARAM_NAMES, sphere_normals, synthetic_envmap
    assert torch.cuda.is_available(), "obsnet_inputs.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    info = gpu_info()
    B, res, thr, He, We = args.batch, 128, float(np.pi / 128 / 2), 1000, 2000

    # inputs
    bank = EnvmapBank(torch.stack([synthetic_envmap(He, We, 500 + b, device=dev, as_numpy=False) for b in range(B)]))
    g = torch.Generator(device=dev).manual_seed(11)
    ids = torch.randperm(B, generator=g, device=dev)
    zK = torch.rand(B, 6, generator=g, device=dev)
    phi = (torch.randint(0, 64, (B,), generator=g, device=dev) / 64.0) * 2 * np.pi - np.pi
    views = torch.stack([torch.sin(phi), torch.zeros_like(phi), torch.cos(phi)], -1)
    n0, m0 = sphere_normals(256)
    n = torch.from_numpy(n0).to(dev)[None].repeat(B, 1, 1, 1)
    n = n + 0.05 * torch.randn(n.shape, generator=g, device=dev)
    inside = torch.from_numpy(m0).to(dev)[None, ..., None]
    nrm_hwc = torch.where(inside, n / n.norm(dim=-1, keepdim=True), torch.zeros((), device=dev))
    normals = nrm_hwc.permute(0, 3, 1, 2).contiguous()  # [B,3,512,512], as ObsNet's renderer returns them
    mask = normals.norm(dim=1) > 0.5
    masked = int(mask.sum())
    renderer = B200RefMapRenderer(res, brdf_param_names=BRDF_PARAM_NAMES)

    def render():
        return render_batch(bank, zK, views, env_index=ids, brdf_param_names=BRDF_PARAM_NAMES, res=res,
                            footprint_S=None, channel_first=True)

    def stitched():
        LrK = render()
        maps, masks = [], []
        for b in range(B):
            nb = normals[b].permute(1, 2, 0)[mask[b]]
            rm, rk = refmap_mask_make(refmap_lookup(LrK[b], nb), nb, res, thr)
            maps.append(rm)
            masks.append(rk)
        raw, raw_mask = torch.stack(maps).permute(0, 3, 1, 2).contiguous(), torch.stack(masks)
        cond, cmask, params = obsnet_condition(raw, raw_mask)
        return cond, cmask, normalized_log_apply(LrK, params), params, raw, raw_mask

    def one_call():
        return obsnet_inputs(renderer, zK, bank, views, normals, mask, env_ids=ids, angle_threshold=thr)[:6]

    # equal outputs, in this run
    a, b = stitched(), one_call()
    flat = lambda o: [t for x in o for t in (x if isinstance(x, tuple) else (x,))]
    equal = all(torch.equal(x, y) for x, y in zip(flat(a), flat(b)))
    print(f"outputs of (a) and (b) equal: {equal} ({masked} masked px in {B} images)")

    def timed(fn):
        dev_ms, wall_ms = [], []
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            wall_ms.append((time.perf_counter() - t0) * 1e3)
            dev_ms.append(e0.elapsed_time(e1))
        return statistics.median(dev_ms), statistics.median(wall_ms)

    # the render alone, which both routes start with: what is left of a route's step is its shading, scatter and
    # conditioning
    routes = {"a_stitched": stitched, "b_obsnet_inputs": one_call, "render_only": render}
    for fn in routes.values():  # warm-up of every shape the timed window uses
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    rounds = []
    for r in range(args.rounds):
        row = {}
        for route, fn in routes.items():
            d, w = timed(fn)
            row[route] = {"device_ms_per_step": round(d, 3), "wall_ms_per_step": round(w, 3)}
        rounds.append(row)
        print(f"round {r}: " + "; ".join(f"{k} {v['device_ms_per_step']:.3f} / {v['wall_ms_per_step']:.3f} ms"
                                          for k, v in row.items()))

    summary = {}
    for key in rounds[0]:
        d = [rw[key]["device_ms_per_step"] for rw in rounds]
        w = [rw[key]["wall_ms_per_step"] for rw in rounds]
        summary[key] = {"device_ms_per_step_min_max": [min(d), max(d)], "wall_ms_per_step_min_max": [min(w), max(w)]}
        if key != "render_only":
            after = [rw[key]["device_ms_per_step"] - rw["render_only"]["device_ms_per_step"] for rw in rounds]
            summary[key]["device_ms_after_render_min_max"] = [round(min(after), 3), round(max(after), 3)]
    result = {
        "what": "ObsNet's training inputs: (a) render_batch + per image compaction, refmap_lookup and refmap_mask_make "
                "+ obsnet_condition + normalized_log_apply vs (b) obsnet_inputs, each step from device tensors to "
                "(cond, mask, LrK transformed, params, raw refmap, raw refmask)",
        "gpu_name_power_limit_max_sm_clock": info, "torch": torch.__version__,
        "inputs": {"samples": B, "envmaps": f"EnvmapBank of {B} synthetic {We}x{He} maps, permuted slots",
                   "normal_maps": "[B,3,512,512], sphere_normals(256), normalise(n + N(0, 0.05)) inside the sphere",
                   "mask": "||n|| > 0.5", "masked_pixels": masked, "res": res, "thr": thr,
                   "footprint": "chosen on the device"},
        "method": f"{args.rounds} rounds alternating (a), (b) and the render alone in one process, {args.steps} steps "
                  "each after 2 warm-up steps; per-step medians; device time = CUDA events around the step, wall = host "
                  "clock around the step and a final synchronise; after render = a route's device time minus the "
                  "render's in the same round",
        "outputs_equal": equal,
        "rounds": rounds, "summary": summary,
    }
    print(f"GPU (name, power limit, max SM clock): {info}")
    for k, v in summary.items():
        print(f"{k}: device {v['device_ms_per_step_min_max']} ms, wall {v['wall_ms_per_step_min_max']} ms per step")
    Path(args.json).parent.mkdir(parents=True, exist_ok=True)
    Path(args.json).write_text(json.dumps(result, indent=1) + "\n")
    if not equal:
        sys.exit("outputs of (a) and (b) differ")


if __name__ == "__main__":
    main()
