#!/usr/bin/env python
"""Benchmarks of the DRMNet rendering hot path on B200 -- BASELINE.json metric and configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload render|img2refmap|synth|sampling] [--batch B] [--footprint auto|S] [--dump-outputs DIR]

workload  (a step is one pass of the hot path over one batch of synthetic input, per GPU; weak scaling over ranks)
  render      BASELINE config[1] -- THE HEADLINE: 64 synthetic 2000x1000 envmaps x random BRDF parameters
              (z ~ U[0,1]^6, dataset/parametricrefmap.py:105; 64 equatorial views, :114-116) -> 64 refmaps of 128x128
  img2refmap  secondary metric (SURVEY 8d): 64 sphere images of 512x512 (~206k masked px each) -> 64 refmaps, res 128
  synth       BASELINE config[2]: training-data synthesis, batch 20 x {LrK, Lrk, Lrkm1} (models/drmnet.py:523-569)
              through callers.synthesize_refmaps (render + luminance normalisation + log transform)
  sampling    BASELINE config[3]: per-step re-render of a sampling batch of 32: r0 -> 128x256 envmap (r0toenvmap,
              models/drmnet.py:931-941) -> render at the current z (DRMNet.reconstruct, :943-952)

value     device-timed whole-job throughput, inputs resident in HBM (larger than L2 for render / img2refmap / synth)
e2e       the same metric through the public API with HOST buffers: pinned inputs copied host->device and the results
          copied back inside the timed region; median of >= 5 steps
roofline  algorithmic bytes of the step / CUDA-event time of the step on the launching stream, against the measured HBM
          copy peak (MEASURED_PEAKS.json).  The render is bound by the FP32 issue rate, not by HBM (DESIGN.md 5): `issue`
          carries the instruction-rate view from the committed ncu captures
cpu_baseline  render: the fp64 oracle port (C + OpenMP, all host cores) on a bounded sample of the same workload;
              img2refmap: the numpy oracle port on one image of the batch (rank 0 only)
Multi-GPU: every rank owns its own envmaps; the rendered refmaps are gathered by ONE equal-count all_gather on a side
stream (drmnet_b200.dist.RefmapGather); `rank_ms` lists every rank's own step time.

--dump-outputs DIR  (e.g. bench_outputs, which git ignores) after the timed steps, rank 0 writes what the last timed
              step returned (the gathered refmaps under multi-GPU) as DIR/<name>.npy, float32 (float64 stays float64).
              The inputs are seeded, so two builds run with the same arguments can be compared array for array.  Past
              64 MB in all, every array is cut to the same seeded sample of its flattened elements and
              DIR/<name>.sample_index.npy holds their positions.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

HE, WE, RES = 1000, 2000, 128
ALG_BYTES_PER_REFMAP = HE * WE * 3 * 4 + RES * RES * 3 * 4 + 40  # SURVEY 8d: 24 196 648
METRICS = {
    "render": ("refmaps rendered/sec (128^2, 2000x1000 envmap)", "refmaps/s"),
    "img2refmap": ("img2refmaps/sec (res 128, ~206k px per image)", "img2refmaps/s"),
    "synth": ("refmaps synthesised/sec (training batch 20 x 3, 2000x1000 envmap, normalised + log)", "refmaps/s"),
    "sampling": ("refmaps re-rendered/sec (sampling batch 32, 128x256 envmap from r0toenvmap)", "refmaps/s"),
}


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


JSON_OUT = sys.stdout  # main() replaces it by a private copy of fd 1


def ncu_summary(workload):
    """Instruction-rate view of the dominant kernel from the committed ncu capture of this workload (profiles/)."""
    p = ROOT / "profiles" / "r2_issue.json"
    try:
        return json.loads(p.read_text()).get(workload)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks and throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# workloads: each returns dict(step=callable -> local result tensor, e2e_step=callable, units=per-rank units per step,
#                              alg_bytes=per-rank algorithmic bytes per step, h2d=, d2h=, config=, dtype=, gather=bool)
# ---------------------------------------------------------------------------------------------------------------------
def footprints(z, mode):
    from drmnet_b200.renderer import auto_footprint, default_alpha_min
    if mode == "auto":
        return [auto_footprint(float(r), RES, default_alpha_min(HE)) for r in z[:, 4].clip(0, 1)]
    return [int(mode)] * z.shape[0]


def wl_render(args, rank, dev):
    import torch
    from drmnet_b200.renderer import render_batch
    from drmnet_b200.synth import sample_brdf, sample_view, synthetic_envmap
    batch = args.batch or 64
    base = 1000 + rank * batch
    envs = torch.empty((batch, HE, WE, 3), dtype=torch.float32, device=dev)
    for b in range(batch):
        envs[b] = synthetic_envmap(HE, WE, seed=base + b, device=dev, as_numpy=False)
    # weak scaling: every rank renders the SAME BRDF / view draws (those of rank 0) on its own envmaps, so the per-GPU work is
    # fixed as N grows (round 1 drew different BRDFs per rank and the rank with the most mirror-like draws set the step)
    z = torch.stack([sample_brdf(1000 + b) for b in range(batch)])
    view = torch.stack([sample_view(1000 + b) for b in range(batch)])
    S_list = footprints(z, args.footprint)
    z_d, view_d = z.to(dev), view.to(dev)
    out = torch.empty((batch, 3, RES, RES), dtype=torch.float32, device=dev)

    def step():
        return render_batch(envs, z_d, view_d, res=RES, footprint_S=S_list, out=out)

    host_envs = envs.cpu().pin_memory()
    host_out = torch.empty((batch, 3, RES, RES), dtype=torch.float32).pin_memory()
    host_z, host_view = z.pin_memory(), view.pin_memory()

    def e2e_step():
        d_env = host_envs.to(dev, non_blocking=True)
        r = render_batch(d_env, host_z.to(dev, non_blocking=True), host_view.to(dev, non_blocking=True), res=RES,
                         footprint_S=S_list)
        host_out.copy_(r, non_blocking=True)
        torch.cuda.synchronize()

    return dict(step=step, e2e_step=e2e_step, units=batch, alg_bytes=batch * ALG_BYTES_PER_REFMAP, gather=True,
                h2d=host_envs.numel() * 4 + host_z.numel() * 4 + host_view.numel() * 4, d2h=host_out.numel() * 4,
                dtype="f32", outputs=lambda r: {"refmaps": r},
                config={"workload": "config[1]: batched parametric refmap render, 64 synthetic 2000x1000 envmaps x random "
                                    "BRDF params -> 128x128 refmaps per GPU (each rank: its own envmaps, the same BRDF / view draws)",
                        "batch_per_gpu": batch,
                        "footprint": args.footprint,
                        "footprint_S_histogram": {str(s): S_list.count(s) for s in sorted(set(S_list))},
                        "l2": "inputs larger than L2 (1.5 GB of envmaps per GPU)"},
                cpu=lambda: cpu_port_sample(batch, 8, args.footprint))


def wl_img2refmap(args, rank, dev):
    import numpy as np
    import torch
    from drmnet_b200.img2refmap import img2refmap_batch
    from drmnet_b200.synth import sphere_image_inputs
    batch = args.batch or 64
    res, thr = 128, float(np.pi / 128 / 2)
    cols, nrms, offs = [], [], [0]
    for b in range(batch):
        c, n = sphere_image_inputs(256, seed=100 + (rank * batch + b) % 8)
        cols.append(c); nrms.append(n); offs.append(offs[-1] + len(c))
    h_col = torch.from_numpy(np.concatenate(cols)).pin_memory()
    h_nrm = torch.from_numpy(np.concatenate(nrms)).pin_memory()
    colors, normals = h_col.to(dev), h_nrm.to(dev)
    offsets = torch.tensor(offs, dtype=torch.int64, device=dev)
    total_n = colors.shape[0]
    h_map = torch.empty((batch, res, res, 3), dtype=torch.float32).pin_memory()
    h_mask = torch.empty((batch, res, res), dtype=torch.bool).pin_memory()

    def step():
        return img2refmap_batch(colors, normals, offsets, res, thr)

    def e2e_step():
        o = img2refmap_batch(h_col.to(dev, non_blocking=True), h_nrm.to(dev, non_blocking=True), offsets, res, thr)
        h_map.copy_(o[0], non_blocking=True)
        h_mask.copy_(o[1], non_blocking=True)
        torch.cuda.synchronize()

    def cpu():
        from oracle.img2refmap_oracle import img2refmap_oracle
        t0 = time.perf_counter()
        img2refmap_oracle(cols[0], nrms[0], res, thr)
        dt = time.perf_counter() - t0
        return 1.0 / dt, dt, 1, (f"numpy port of utils/img2refmap.py:6-37 (oracle/img2refmap_oracle.py), one image of the "
                                 f"batch ({len(cols[0])} px) in {dt:.2f} s; the reference's own O(res^2 n) torch code took "
                                 "3.6 s on 8 cores for a 27 774-px image (BASELINE.md)")

    return dict(step=step, e2e_step=e2e_step, units=batch, alg_bytes=24 * total_n + batch * res * res * (13 + 8),
                gather=False, h2d=(h_col.numel() + h_nrm.numel()) * 4, d2h=h_map.numel() * 4 + h_mask.numel(),
                dtype="f32 compare / u32 keys",
                outputs=lambda r: {"refmap": r[0], "refmask": r[1], "counts": r[2], "sel_index": r[3]},
                config={"workload": "img2refmap: 64 sphere images of 512x512 (SURVEY 8d inputs (b),(c)) -> 64 refmaps, "
                                    "res 128, thr pi/256", "batch_per_gpu": batch, "pixels_per_image": total_n // batch,
                        "l2": "inputs larger than L2 (317 MB of pixels per GPU)"},
                cpu=cpu)


def wl_synth(args, rank, dev):
    import torch
    from drmnet_b200.callers import synthesize_refmaps
    from drmnet_b200.renderer import B200RefMapRenderer
    from drmnet_b200.synth import BRDF_PARAM_NAMES, sample_brdf, sample_view, schedule_point, synthetic_envmap
    B = args.batch or 20
    base = 2000 + rank * B
    envs = torch.stack([synthetic_envmap(HE, WE, base + b, device=dev, as_numpy=False) for b in range(B)])
    zK = torch.stack([sample_brdf(base + b) for b in range(B)])
    sched = [schedule_point(zK[b], float(torch.rand((), generator=torch.Generator().manual_seed(base + b)))) for b in range(B)]
    stacked_z = torch.stack([zK, torch.stack([s[2] for s in sched]).float(), torch.stack([s[3] for s in sched]).float()])
    views = torch.stack([sample_view(base + b) for b in range(B)])
    r = B200RefMapRenderer(refmap_res=RES, spp=256, denoise="simple", brdf_param_names=BRDF_PARAM_NAMES)
    h_env = envs.cpu().pin_memory()
    h_out = torch.empty((3, B, 3, RES, RES), dtype=torch.float32).pin_memory()

    def step():
        post, scale, raw = synthesize_refmaps(r, stacked_z, envs, views)
        return torch.stack(post), scale, raw

    def e2e_step():
        o = synthesize_refmaps(r, stacked_z, h_env.to(dev, non_blocking=True), views)[0]
        h_out.copy_(torch.stack(o), non_blocking=True)
        torch.cuda.synchronize()

    return dict(step=step, e2e_step=e2e_step, units=3 * B, alg_bytes=B * HE * WE * 12 + 3 * B * (RES * RES * 12 + 40),
                gather=False, h2d=h_env.numel() * 4, d2h=h_out.numel() * 4, dtype="f32",
                outputs=lambda o: {"refmaps": o[0], "normalizing_scale": o[1], "raw": o[2]},
                config={"workload": "config[2]: training-data synthesis, batch 20 x {LrK, Lrk, Lrkm1} sharing envmap and "
                                    "view, render + luminance normalisation + log transform", "batch_per_gpu": B,
                        "renders_per_step_per_gpu": 3 * B, "l2": "inputs larger than L2 (480 MB of envmaps per GPU)"},
                cpu=None)


def wl_sampling(args, rank, dev):
    import torch
    from drmnet_b200.callers import r0toenvmap
    from drmnet_b200.renderer import render_batch
    from drmnet_b200.synth import Z0, sample_brdf, synthetic_envmap
    B = args.batch or 32
    one = torch.tensor([[0.0, 0.0, 1.1]])
    basis = render_batch(torch.ones(1, 128, 256, 3, device=dev), torch.tensor([list(Z0)]), one, res=RES, footprint_S=2)[0]
    env0 = synthetic_envmap(HE, WE, 3000 + rank, device=dev, as_numpy=False)[None]
    r0 = render_batch(env0, torch.tensor([list(Z0)]), one, res=RES, footprint_S=4).expand(B, 3, RES, RES).contiguous()
    z = torch.stack([sample_brdf(3000 + rank * B + b) for b in range(B)]).to(dev)
    view = one.expand(B, 3).contiguous().to(dev)
    rough = z[:, 4].clip(0, 1).tolist()
    from drmnet_b200.renderer import auto_footprint, default_alpha_min
    S_list = [auto_footprint(r, RES, default_alpha_min(128)) for r in rough]
    h_r0 = r0.cpu().pin_memory()
    h_out = torch.empty((B, 3, RES, RES), dtype=torch.float32).pin_memory()

    def step():
        env = r0toenvmap(r0, basis.clamp_min(1e-3), (128, 256)).contiguous()
        return render_batch(env, z, view, res=RES, footprint_S=S_list)

    def e2e_step():
        env = r0toenvmap(h_r0.to(dev, non_blocking=True), basis.clamp_min(1e-3), (128, 256)).contiguous()
        h_out.copy_(render_batch(env, z, view, res=RES, footprint_S=S_list), non_blocking=True)
        torch.cuda.synchronize()

    return dict(step=step, e2e_step=e2e_step, units=B, alg_bytes=B * (RES * RES * 12 * 2 + 128 * 256 * 12 * 2), gather=True,
                h2d=h_r0.numel() * 4, d2h=h_out.numel() * 4, dtype="f32", outputs=lambda r: {"refmaps": r},
                config={"workload": "config[3]: per-step re-render of a sampling batch of 32 (r0toenvmap -> 128x256 envmap -> "
                                    "render at the current z); the U-Nets are stock PyTorch and not part of the step",
                        "batch_per_gpu": B, "l2": "flushed between steps (a 256 MB buffer is written)"},
                cpu=None, flush_l2=True)


WORKLOADS = {"render": wl_render, "img2refmap": wl_img2refmap, "synth": wl_synth, "sampling": wl_sampling}

_CPU_ENV = None


def cpu_port_sample(batch, n_renders, footprint):
    """The fp64 oracle port (C + OpenMP, all host cores) on a bounded sample of the render workload: the first
    `n_renders` renders of rank 0's batch, each with its own footprint S, each on a k x k block of cells of the 128x128
    refmap sized so one render costs about a second (cost ~ cells x S^2 x texels).  refmaps/s = sum(cell fractions) /
    sum(times)."""
    from drmnet_b200.renderer import auto_footprint, default_alpha_min
    from drmnet_b200.synth import sample_brdf, sample_view, synthetic_envmap
    from oracle import render_oracle as ro
    ro.build()
    ro.set_threads(os.cpu_count() or 1)
    global _CPU_ENV
    if _CPU_ENV is None:
        _CPU_ENV = synthetic_envmap(HE, WE, seed=1000)
    env = _CPU_ENV
    frac_sum, t_sum, desc = 0.0, 0.0, []
    for b in range(n_renders):
        z = sample_brdf(1000 + b % batch)
        S = auto_footprint(float(z[4]), RES, default_alpha_min(HE)) if footprint == "auto" else int(footprint)
        k = max(1, 24 // S)
        i0 = (RES - k) // 2
        t0 = time.perf_counter()
        ro.render_oracle(env, z.tolist(), sample_view(1000 + b % batch).tolist(), RES, S=S, window=(i0, i0 + k, i0, i0 + k))
        t_sum += time.perf_counter() - t0
        frac_sum += (k * k) / float(RES * RES)
        desc.append(f"S={S}:{k}x{k}")
    return frac_sum / t_sum, t_sum, ro.num_threads(), (
        f"fp64 oracle port (C + OpenMP), first {n_renders} renders of the batch with their own footprint S on a centred k x k "
        f"block of the 128x128 cells over the full 2000x1000 envmap [{', '.join(desc)}]: {frac_sum:.5f} refmap in {t_sum:.1f} s")


def run_reference(args):
    """--impl reference: the reference has no CPU renderer (Mitsuba cuda_ad_rgb is hard-coded, main.py:26) and Mitsuba
    is unavailable; the timed arm is the oracle port on all host threads, each step a bounded sample of the workload.
    For img2refmap the port is the numpy restatement of utils/img2refmap.py."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    metric, unit = METRICS[args.workload]
    vals, ms, cores, sample = [], [], 1, ""
    for it in range(args.warmup + args.steps):
        if args.workload == "img2refmap":
            import numpy as np
            from drmnet_b200.synth import sphere_image_inputs
            from oracle.img2refmap_oracle import img2refmap_oracle
            c, n = sphere_image_inputs(256, seed=100)
            t0 = time.perf_counter()
            img2refmap_oracle(c, n, 128, float(np.pi / 256))
            t = time.perf_counter() - t0
            v, cores, sample = 1.0 / t, 1, f"numpy port of utils/img2refmap.py, one image of {len(c)} px per step"
        else:
            v, t, cores, sample = cpu_port_sample(args.batch or 64, 4, args.footprint)
        if it >= args.warmup:
            vals.append(v); ms.append(t * 1e3)
    value = sum(vals) / len(vals)
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sum(ms) / len(ms), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload} (bounded sample per step on the host cores)", "footprint": args.footprint},
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), file=JSON_OUT, flush=True)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(arrays, out_dir):
    """Write {name: tensor} as out_dir/<name>.npy in float32 (float64 kept).  When the arrays exceed DUMP_LIMIT_BYTES
    together, each keeps the same fraction of its flattened elements, drawn with a fixed seed, and
    out_dir/<name>.sample_index.npy (float64) lists which."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        host[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    frac = 1.0
    if sum(a.nbytes for a in host.values()) > DUMP_LIMIT_BYTES:
        # a sampled element costs its value plus a float64 index; 4 KB per file covers the .npy headers
        budget = DUMP_LIMIT_BYTES - 4096 * 2 * len(host)
        frac = budget / sum(a.size * (a.itemsize + 8) for a in host.values())
    for name, a in host.items():
        if frac < 1.0:
            idx = np.sort(np.random.default_rng(0).choice(a.size, max(1, int(a.size * frac)), replace=False))
            np.save(out_dir / f"{name}.sample_index.npy", idx.astype(np.float64))
            a = a.reshape(-1)[idx]
        np.save(out_dir / f"{name}.npy", a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="render", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="units per GPU per step (0: the workload's own: 64 / 64 / 20 / 32)")
    ap.add_argument("--footprint", default="auto", help="'auto' (per render, from its roughness) or 1, 2, 4, 8, 16")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries the JSON line and nothing else: whatever libraries print there (NCCL's version banner at init)
    # goes to stderr
    global JSON_OUT
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from drmnet_b200 import _lib
    from drmnet_b200.dist import RefmapGather

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU path"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    W = WORKLOADS[args.workload](args, rank, dev)
    units = W["units"]
    gather = None
    if world > 1 and W["gather"]:
        ids = [torch.arange(units) + r * units for r in range(world)]  # a pure function of the rank: no count exchange
        gather = RefmapGather(ids, units * world, dev)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev) if W.get("flush_l2") else None

    def step():
        if flush is not None:
            flush.zero_()
        r = W["step"]()
        if gather is not None:
            gather.launch(r)  # side stream: the next step's kernels start while the blocks travel
        return r

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        last = step()  # held like the timed loop holds it, so the allocator is warmed for the same footprint
    if gather is not None:
        gather.result()
    barrier()
    launches0 = L.drm_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev[0].record()
        for i in range(args.steps):
            last = step()
            ev[i + 1].record()
        if gather is not None:
            last = gather.result()
            end = torch.cuda.Event(enable_timing=True)
            end.record()
        else:
            end = ev[-1]
        barrier()
    launches = L.drm_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        # before anything else runs: the render writes every step into the same buffer
        dump_outputs(W["outputs"](last), args.dump_outputs)
    clock_info = clocks.summary()
    if clock_info["samples"] < 2:
        # the timed region was shorter than nvidia-smi's sampling period: keep the same load running until it has sampled
        with ClockSampler(local_rank) as clocks2:
            t_end = time.perf_counter() + 0.9
            while time.perf_counter() < t_end:
                step()
                torch.cuda.synchronize()
            if gather is not None:
                gather.result()
        clock_info = dict(clocks2.summary(), note="timed region shorter than the 200 ms sampling period: sampled while "
                                                  "the same steps kept running right after it")
    ms_own = ev[0].elapsed_time(end)
    ms_compute = ev[0].elapsed_time(ev[-1])  # this rank's own kernels, before it waits for the other ranks' blocks
    t = torch.tensor([ms_own, ms_compute], dtype=torch.float64, device=dev)
    all_ms = [t.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(all_ms, t)
    rank_ms = [float(x[0].item()) / args.steps for x in all_ms]
    rank_compute_ms = [float(x[1].item()) / args.steps for x in all_ms]
    ms = max(float(x[0].item()) for x in all_ms)
    ms_per_step = ms / args.steps
    value = units * world * args.steps / (ms / 1e3)

    # ---- end to end through the public API with host buffers (pinned), H2D + D2H inside the timed region -------------
    W["e2e_step"]()
    barrier()
    e2e_times = []
    for _ in range(max(5, args.e2e_steps)):
        barrier()
        t0 = time.perf_counter()
        W["e2e_step"]()
        barrier()
        e2e_times.append(time.perf_counter() - t0)
    e2e_s = torch.tensor([statistics.median(e2e_times)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = units * world / float(e2e_s.item())

    if rank == 0:
        metric, unit = METRICS[args.workload]
        peak, peak_src = hbm_peak()
        achieved = W["alg_bytes"] / (rank_ms[0] / 1e3) / 1e9
        line = {
            "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": W["dtype"], "data": "synthetic",
            "config": dict(W["config"], parallelism=f"dp{world}",
                           collective="one equal-count all_gather of the results on a side stream" if gather else "none"),
            "rank_ms": {"per_rank": rank_ms, "min": min(rank_ms), "max": max(rank_ms),
                        "compute_only_per_rank": rank_compute_ms,
                        "note": "per_rank includes waiting for the gathered blocks of the slowest rank; compute_only is the "
                                "rank's own kernels"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (ncu_summary(args.workload) or {}).get("dram_bytes_per_step"),
                         "algorithmic_bytes_per_step": W["alg_bytes"], "peak_source": peak_src,
                         "note": "whole step (every launch) on the launching stream; the render is bound by the FP32 issue rate, "
                                 "not by HBM (DESIGN.md 5)" if args.workload != "img2refmap" else
                                 "whole step (every launch) on the launching stream"},
            "issue": ncu_summary(args.workload),
            "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": W["h2d"], "d2h_bytes_per_step": W["d2h"],
                    "steps": len(e2e_times), "statistic": "median"},
            "gpu_launches": int(launches),
            "clocks": clock_info,
        }
        if not args.no_cpu_baseline and W.get("cpu"):
            v, _, cores, sample = W["cpu"]()
            line["cpu_baseline"] = {"value": v, "unit": unit, "cores": cores, "kind": "port", "sample": sample}
        print(json.dumps(line), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
