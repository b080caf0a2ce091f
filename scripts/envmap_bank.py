"""What envmap banks save: diffuse pyramids built once per map instead of once per render call (GPU).

    python scripts/envmap_bank.py [--rounds R] [--steps K] [--bank B] [--json FILE]

Old and new paths alternate R times in one process, and the card's name and power limit are read in the same run:
  1. The drop-in loop as DRMNet's get_input issues it, on the inputs of `bench.py --workload synth` (20 fp32 2000 x 1000
     maps, seeds 2000..2019, 3 BRDF vectors per map): per map, `rendering(envmap=map)` and then `rendering()` twice.
     Old: every call renders its map through render_batch, which builds the map's diffuse pyramid.  New:
     B200RefMapRenderer, which keeps the map as a bank of one.  CUDA events around each call and around the step.
  2. A training-like step of 64 renders (the BRDF and view draws of `bench.py --workload render`) drawn from a
     resident bank of B fp16 2000 x 1000 maps.  New: render_batch on the bank with env_index = the drawn slots.  Old:
     the 64 maps copied host to device from pinned memory, then render_batch on them, synchronised (host clock).  The
     kernel-only old step (the 64 maps already resident) is timed too.  The bank render is checked to be bit-identical
     to the old one.
  3. The pyramid build per map (the whole bank) and the update of 64 slots (re-read in place, and copied from device
     maps).
  4. Workspace bytes of both render paths at B = 64 and 1024, and the bank's pyramid bytes.
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
    ap.add_argument("--bank", type=int, default=1024)
    ap.add_argument("--json", default=str(ROOT / "profiles" / "r6_envmap_bank.json"))
    args = ap.parse_args()
    if args.rounds < 3 or args.steps < 1 or args.bank < 64:
        ap.error("--rounds >= 3, --steps >= 1, --bank >= 64")

    import torch

    import bench
    from drmnet_b200 import _lib
    from drmnet_b200.renderer import B200RefMapRenderer, EnvmapBank, render_batch
    from drmnet_b200.synth import BRDF_PARAM_NAMES, sample_brdf, sample_view, schedule_point, synthetic_envmap
    assert torch.cuda.is_available(), "envmap_bank.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info()
    L = _lib.lib()
    HE, WE, RES = bench.HE, bench.WE, bench.RES

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    # ---- 1. the drop-in loop of get_input -----------------------------------------------------------------------------
    B, base = 20, 2000  # bench.wl_synth on rank 0
    envs = torch.stack([synthetic_envmap(HE, WE, base + b, device=dev, as_numpy=False) for b in range(B)])
    zK = torch.stack([sample_brdf(base + b) for b in range(B)])
    sched = [schedule_point(zK[b], float(torch.rand((), generator=torch.Generator().manual_seed(base + b))))
             for b in range(B)]
    stacked_z = torch.stack([zK, torch.stack([s[2] for s in sched]).float(), torch.stack([s[3] for s in sched]).float()])
    views = torch.stack([sample_view(base + b) for b in range(B)])
    renderers = {"old": B200RefMapRenderer(refmap_res=RES, brdf_param_names=BRDF_PARAM_NAMES),
                 "new": B200RefMapRenderer(refmap_res=RES, brdf_param_names=BRDF_PARAM_NAMES)}
    old = renderers["old"]
    old._persistent_bank = lambda: old._envmap  # the parent's call: render_batch(map[None]) builds the pyramid

    def drop_in_step(r, marks=None):
        outs = []
        for b in range(B):
            for g in range(3):
                a = ev() if marks is not None else None
                outs.append(r.rendering(stacked_z[g, b], BRDF_PARAM_NAMES, envmap=envs[b] if g == 0 else None,
                                        view_from=views[b] if g == 0 else None))
                if marks is not None:
                    marks.append((g, a, ev()))
        return outs

    outs = {k: drop_in_step(r) for k, r in renderers.items()}  # warm-up and the check
    torch.cuda.synchronize()
    drop_in_equal = all(torch.equal(x, y) for x, y in zip(outs["old"], outs["new"]))
    del outs
    launches = {}
    for k, r in renderers.items():
        n0 = L.drm_launch_count()
        drop_in_step(r)
        launches[k] = (L.drm_launch_count() - n0) / (3 * B)
    drop_in = {k: {"ms_per_step": [], "ms_per_call_with_envmap": [], "ms_per_call_envmap_none": []} for k in renderers}
    for _ in range(args.rounds):
        for k, r in renderers.items():
            torch.cuda.synchronize()
            a = ev()
            drop_in_step(r)
            b = ev()
            torch.cuda.synchronize()
            drop_in[k]["ms_per_step"].append(a.elapsed_time(b))
            marks = []
            drop_in_step(r, marks)
            torch.cuda.synchronize()
            first = [s.elapsed_time(e) for g, s, e in marks if g == 0]
            rest = [s.elapsed_time(e) for g, s, e in marks if g > 0]
            drop_in[k]["ms_per_call_with_envmap"].append(statistics.median(first))
            drop_in[k]["ms_per_call_envmap_none"].append(statistics.median(rest))
    for k in drop_in:
        drop_in[k]["launches_per_call"] = launches[k]
    del envs, renderers, old
    torch.cuda.empty_cache()

    # ---- 2. a training step of 64 renders from a resident bank --------------------------------------------------------
    nb, batch = args.bank, 64
    maps = torch.empty((nb, HE, WE, 3), dtype=torch.float16, device=dev)
    for b in range(nb):
        maps[b] = synthetic_envmap(HE, WE, seed=10000 + b, device=dev, as_numpy=False).clamp(max=65504).half()
    torch.cuda.synchronize()
    # 3. (first) the build of the whole bank
    build_ms = []
    for i in range(args.rounds):
        torch.cuda.synchronize()
        a = ev()
        bank = EnvmapBank(maps)
        b = ev()
        torch.cuda.synchronize()
        build_ms.append(a.elapsed_time(b))
    z = torch.stack([sample_brdf(1000 + b) for b in range(batch)])
    view = torch.stack([sample_view(1000 + b) for b in range(batch)])
    S_list = bench.footprints(z, "auto")
    slots = torch.randperm(nb, generator=torch.Generator().manual_seed(6))[:batch]
    slots_d = slots.to(dev, torch.int32)
    z_d, view_d = z.to(dev), view.to(dev)
    host_maps = maps[slots.to(dev)].cpu().pin_memory()
    host_out = torch.empty((batch, 3, RES, RES), dtype=torch.float32).pin_memory()
    resident = maps[slots.to(dev)].contiguous()

    def new_step():
        r = render_batch(bank, z_d, view_d, env_index=slots_d, res=RES, footprint_S=S_list)
        host_out.copy_(r, non_blocking=True)
        torch.cuda.synchronize()
        return r

    def old_step():
        d_env = host_maps.to(dev, non_blocking=True)
        r = render_batch(d_env, z_d, view_d, res=RES, footprint_S=S_list)
        host_out.copy_(r, non_blocking=True)
        torch.cuda.synchronize()
        return r

    def old_kernel_step():
        return render_batch(resident, z_d, view_d, res=RES, footprint_S=S_list)

    bank_equal = bool(torch.equal(new_step(), old_step()))
    old_kernel_step()
    train = {"new_bank_ms": [], "old_h2d_render_ms": [], "old_resident_kernel_ms": []}
    for _ in range(args.rounds):
        for key, fn in (("new_bank_ms", new_step), ("old_h2d_render_ms", old_step)):
            for _ in range(args.steps):
                t0 = time.perf_counter()
                fn()
                train[key].append(1e3 * (time.perf_counter() - t0))
        torch.cuda.synchronize()
        a = ev()
        for _ in range(args.steps):
            old_kernel_step()
        b = ev()
        torch.cuda.synchronize()
        train["old_resident_kernel_ms"].append(a.elapsed_time(b) / args.steps)
    # 3. update 64 slots: re-read in place, and copied in from device maps
    upd = {"update_64_in_place_ms": [], "update_64_copy_ms": []}
    new_maps = resident.flip(0).contiguous()
    ids = slots.tolist()
    for _ in range(args.rounds):
        torch.cuda.synchronize()
        a = ev()
        bank.update(ids)
        b = ev()
        torch.cuda.synchronize()
        upd["update_64_in_place_ms"].append(a.elapsed_time(b))
        a = ev()
        bank.update(ids, new_maps)
        b = ev()
        torch.cuda.synchronize()
        upd["update_64_copy_ms"].append(a.elapsed_time(b))

    # ---- 4. workspace bytes ---------------------------------------------------------------------------------------------
    ws = {str(n): {"render_workspace_bytes": L.drm_render_workspace_bytes(batch, n, HE, WE, RES, 0),
                   "prepared_workspace_bytes": L.drm_render_prepared_workspace_bytes(batch, n, HE, WE, RES, 0),
                   "bank_pyramid_bytes": L.drm_env_pyramid_bytes(n, HE, WE)} for n in (64, 1024)}

    med = {k: statistics.median(v) for k, v in train.items()}
    result = {
        "gpu_name_power_limit_max_sm_clock": info, "torch": torch.__version__,
        "drop_in_get_input_loop": {"maps": B, "calls_per_map": 3, "envmap": [HE, WE], "dtype": "fp32", "refmap_res": RES,
                                   "bit_identical": drop_in_equal, **drop_in},
        "training_step": {"bank_maps": nb, "dtype": "fp16", "renders": batch,
                          "footprint_S_histogram": {str(s): S_list.count(s) for s in sorted(set(S_list))},
                          "bit_identical": bank_equal, "ms_all": train, "ms_median": med,
                          "refmaps_per_s": {k: batch / (v / 1e3) for k, v in med.items()},
                          "h2d_bytes_old": host_maps.numel() * 2, "h2d_bytes_new": 0},
        "build": {"bank_build_ms": build_ms, "ms_per_map": min(build_ms) / nb, **upd},
        "workspace": ws,
    }
    print(f"GPU (name, power limit, max SM clock): {info}")
    for k in ("old", "new"):
        d = drop_in[k]
        print(f"drop-in {k}: step {', '.join(f'{t:.1f}' for t in d['ms_per_step'])} ms; per call with envmap "
              f"{statistics.median(d['ms_per_call_with_envmap']):.3f} ms, envmap=None "
              f"{statistics.median(d['ms_per_call_envmap_none']):.3f} ms; {d['launches_per_call']:.1f} launches/call")
    print(f"drop-in bit-identical: {drop_in_equal}")
    print(f"training step (64 of {nb} fp16 maps): " + ", ".join(f"{k} {v:.1f}" for k, v in med.items())
          + f"; bit-identical: {bank_equal}")
    print(f"bank build {min(build_ms):.1f} ms = {min(build_ms) / nb:.3f} ms/map; update 64 in place "
          f"{min(upd['update_64_in_place_ms']):.2f} ms, copied {min(upd['update_64_copy_ms']):.2f} ms")
    print(f"workspace: {ws}")
    Path(args.json).parent.mkdir(parents=True, exist_ok=True)
    Path(args.json).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
