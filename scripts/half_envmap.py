"""What rendering from fp16 envmaps costs and saves on the bench's render inputs (GPU).

    python scripts/half_envmap.py [--rounds R] [--steps K] [--e2e-steps E] [--json FILE]

Inputs are those of `bench.py --workload render`: 64 synthetic 2000 x 1000 envmaps (seeds 1000..1063), the same BRDF
and view draws, auto footprints, 128^2 refmaps.  The fp16 maps are `env.clamp(max=65504).half()`.  It measures, in one
process:
  1. kernel time per step with the maps resident on the device, fp32 and fp16 alternated R times (CUDA events around K
     steps each);
  2. the end-to-end step from pinned host memory as bench.py's e2e_step does it (H2D of maps, BRDFs and views, render,
     D2H of the refmaps, synchronise), fp32 and fp16 alternated R times, E host-timed steps each, median over all;
  3. the accuracy cost of storing the maps in fp16: render(env) against render(env.half()), relative L2 per refmap
     and the worst cell, next to the quantisation error of the maps themselves;
and checks that render(env.half()) is bit-identical to render(env.half().float()).  The card's name and power limit
are read in the same run.
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
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--json", default=str(ROOT / "profiles" / "r5_half_envmap.json"))
    args = ap.parse_args()
    if args.rounds < 3 or args.steps < 1 or args.e2e_steps < 5:
        ap.error("--rounds >= 3, --steps >= 1, --e2e-steps >= 5")

    import torch

    import bench
    from drmnet_b200.renderer import render_batch
    from drmnet_b200.synth import sample_brdf, sample_view, synthetic_envmap
    assert torch.cuda.is_available(), "half_envmap.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info()

    batch, base = 64, 1000  # bench.wl_render on rank 0
    env32 = torch.empty((batch, bench.HE, bench.WE, 3), dtype=torch.float32, device=dev)
    for b in range(batch):
        env32[b] = synthetic_envmap(bench.HE, bench.WE, seed=base + b, device=dev, as_numpy=False)
    clamped = int((env32 > 65504).sum())
    env16 = env32.clamp(max=65504).half()
    z = torch.stack([sample_brdf(base + b) for b in range(batch)])
    view = torch.stack([sample_view(base + b) for b in range(batch)])
    S_list = bench.footprints(z, "auto")
    z_d, view_d = z.to(dev), view.to(dev)
    shape = (batch, 3, bench.RES, bench.RES)
    envs = {"fp32": env32, "fp16": env16}
    outs = {k: torch.empty(shape, dtype=torch.float32, device=dev) for k in envs}

    def step(k):
        return render_batch(envs[k], z_d, view_d, res=bench.RES, footprint_S=S_list, out=outs[k])

    # ---- 3 first (also the warm-up): accuracy and bit identity ------------------------------------------------------
    for k in envs:
        step(k)
    up = render_batch(env16.float(), z_d, view_d, res=bench.RES, footprint_S=S_list)
    torch.cuda.synchronize()
    bit_identical = bool(torch.equal(outs["fp16"], up))
    del up
    ref, q = outs["fp32"].double(), outs["fp16"].double()
    d = (q - ref).flatten(1)
    rel_l2 = (d.norm(dim=1) / ref.flatten(1).norm(dim=1)).cpu()
    cell_d = (q - ref).norm(dim=1)                       # [N, res, res]: per-cell RGB difference
    cell_r = ref.norm(dim=1)
    peak = cell_r.flatten(1).max(dim=1).values[:, None, None]
    worst_cell_rel_peak = float((cell_d / peak).max())   # worst cell, relative to its refmap's brightest cell
    lit = cell_r > 1e-3 * peak
    worst_cell_rel = float((cell_d[lit] / cell_r[lit]).max())  # ... relative to the cell itself (cells above 1e-3 peak)
    e32 = env32.double().flatten(1)
    env_rel_l2 = ((env16.double().flatten(1) - e32).norm(dim=1) / e32.norm(dim=1)).cpu()
    accuracy = {"refmap_rel_l2": {"max": float(rel_l2.max()), "median": float(rel_l2.median()),
                                  "min": float(rel_l2.min())},
                "worst_cell_rel_to_refmap_peak": worst_cell_rel_peak,
                "worst_cell_rel_to_itself_above_1e-3_peak": worst_cell_rel,
                "envmap_rel_l2": {"max": float(env_rel_l2.max()), "median": float(env_rel_l2.median())},
                "texels_clamped_at_65504": clamped}
    del ref, q, d, cell_d, cell_r, lit, e32

    # ---- 1. kernel time per step, resident maps -----------------------------------------------------------------------
    kernel = {k: [] for k in envs}
    for _ in range(args.rounds):
        for k in envs:
            step(k)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(args.steps):
                step(k)
            b.record()
            torch.cuda.synchronize()
            kernel[k].append(a.elapsed_time(b) / args.steps)

    # ---- 2. end-to-end step from pinned host memory (bench.wl_render's e2e_step) --------------------------------------
    host = {k: v.cpu().pin_memory() for k, v in envs.items()}
    del envs, env32, env16
    torch.cuda.empty_cache()
    host_z, host_view = z.pin_memory(), view.pin_memory()
    host_out = torch.empty(shape, dtype=torch.float32).pin_memory()

    def e2e_step(k):
        d_env = host[k].to(dev, non_blocking=True)
        r = render_batch(d_env, host_z.to(dev, non_blocking=True), host_view.to(dev, non_blocking=True), res=bench.RES,
                         footprint_S=S_list)
        host_out.copy_(r, non_blocking=True)
        torch.cuda.synchronize()

    e2e = {k: [] for k in host}
    for k in host:
        e2e_step(k)
    for _ in range(args.rounds):
        for k in host:
            for _ in range(args.e2e_steps):
                t0 = time.perf_counter()
                e2e_step(k)
                e2e[k].append(1e3 * (time.perf_counter() - t0))
    h2d = {k: host[k].numel() * host[k].element_size() + host_z.numel() * 4 + host_view.numel() * 4 for k in host}

    result = {"gpu_name_power_limit_max_sm_clock": info, "torch": torch.__version__, "renders_per_step": batch,
              "envmap": [bench.HE, bench.WE], "refmap_res": bench.RES,
              "footprint_S_histogram": {str(s): S_list.count(s) for s in sorted(set(S_list))},
              "fp16_bit_identical_to_fp32_upcast": bit_identical, "accuracy_fp16_storage": accuracy}
    for k in ("fp32", "fp16"):
        med = statistics.median(e2e[k])
        result[k] = {"kernel_ms_per_step_rounds": kernel[k], "kernel_refmaps_per_s": batch / (min(kernel[k]) / 1e3),
                     "e2e_ms_per_step_all": e2e[k], "e2e_ms_per_step_median": med,
                     "e2e_refmaps_per_s": batch / (med / 1e3), "h2d_bytes_per_step": h2d[k],
                     "d2h_bytes_per_step": host_out.numel() * 4}
    print(f"GPU (name, power limit, max SM clock): {info}")
    for k in ("fp32", "fp16"):
        r = result[k]
        print(f"{k}: kernel {', '.join(f'{t:.1f}' for t in r['kernel_ms_per_step_rounds'])} ms/step; e2e median "
              f"{r['e2e_ms_per_step_median']:.1f} ms/step = {r['e2e_refmaps_per_s']:.1f} refmaps/s; "
              f"H2D {r['h2d_bytes_per_step'] / 1e9:.3f} GB/step")
    print(f"fp16 render == fp32 render of the upcast map: {bit_identical}")
    print(f"fp16 storage: refmap rel-L2 max {accuracy['refmap_rel_l2']['max']:.2e} median "
          f"{accuracy['refmap_rel_l2']['median']:.2e}; worst cell {worst_cell_rel_peak:.2e} of its refmap's peak, "
          f"{worst_cell_rel:.2e} of itself; envmap rel-L2 max {accuracy['envmap_rel_l2']['max']:.2e}")
    Path(args.json).parent.mkdir(parents=True, exist_ok=True)
    Path(args.json).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
