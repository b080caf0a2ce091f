"""Per-pass traversal statistics of one render per footprint class (development tool, GPU).

Besides the traversal counts, every specular pass reports the share of its warps' cycles spent in the barriers of the
item loop, waiting for the slowest warp of their 16 x 16-node tile (status words 50.. and 56.. of the workspace)."""
import ctypes
import sys
from pathlib import Path
import torch
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from drmnet_b200 import _lib
from drmnet_b200.synth import synthetic_envmap
STAT_TILE_WAIT, STAT_WARP_CYCLES = 50, 56


def render_stats(env, z, v, opts, res=128):
    """One render with collect_stats; returns the 64 status words of its workspace."""
    L = _lib.lib()
    _, He, We, _ = env.shape
    nbytes = L.drm_render_workspace_bytes(1, 1, He, We, res, 0)
    ws = torch.zeros(int(nbytes), dtype=torch.uint8, device=env.device)
    out = torch.empty((1, 3, res, res), dtype=torch.float32, device=env.device)
    idx = torch.zeros(1, dtype=torch.int32, device=env.device)
    z, v = z.to(env.device).contiguous(), v.to(env.device).contiguous()
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(L.drm_render_refmaps_opts(env.data_ptr(), 1, He, We, idx.data_ptr(), z.data_ptr(), v.data_ptr(), None, 1,
                                         res, 0, 0.0, 1, out.data_ptr(), ws.data_ptr(), ws.numel(), stream,
                                         ctypes.byref(opts)))
    torch.cuda.synchronize()
    st = ws[:256].view(torch.int32).tolist()
    if st[0]:
        raise RuntimeError(f"render status {st[0]}")
    return st


env = torch.from_numpy(synthetic_envmap(1000, 2000, seed=1001)).cuda()[None].contiguous()
v = torch.tensor([[0.3, 0.0, 1.0]])
for rough in [float(x) for x in sys.argv[1:]] or [0.7, 0.3, 0.15, 0.09, 0.0]:
    for name, kw in (("default", {}), ("rim off", {"limb_x": 0.0})):
        o = _lib.default_render_options(); o.collect_stats = 1
        for k, val in kw.items(): setattr(o, k, val)
        z = torch.tensor([[0.5, 0.9, 0.5, 0.3, rough, 1.0]])
        st = render_stats(env, z, v, o)
        print(f"rough {rough} [{name}]")
        for p in range(5):
            vis, it, a0, a1 = st[16 + 4 * p: 20 + 4 * p]
            if vis:
                wait, cyc = st[STAT_TILE_WAIT + p], st[STAT_WARP_CYCLES + p]
                print(f"  pass {p}: visits {vis/1e6:7.2f} M  iters {it/1e6:6.2f} M (fill {vis/max(it,1)/32:.2f})  texel recs {a0/1e6:7.2f} M  pyramid recs {a1/1e6:7.2f} M"
                      f"  -> per cell: visits {vis*32/16384:9.0f} pairs0 {a0*32/16384:9.0f} pairs1 {a1*32/16384:9.0f}"
                      f"  tile wait {100 * wait / max(cyc, 1):5.1f} % of warp cycles")
