"""fp16 environment maps.  The tree render reads fp16 texels in place and converts them where it loads them; the
conversion is exact and nothing after the load differs, so every render of an fp16 map must be bit-identical to the
render of the same map upcast to fp32: every lattice, several launch sequences, the sampling map size, the drop-in
renderer and the batched callers."""
import ctypes
import math

import pytest
import torch

from drmnet_b200 import _lib
from drmnet_b200.callers import rendering_refmaps, synthesize_refmaps
from drmnet_b200.renderer import B200RefMapRenderer, render_batch
from drmnet_b200.synth import BRDF_PARAM_NAMES, Z0, sample_brdf, sample_view, synthetic_envmap

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
VIEWS = [[0.0, 0.0, 1.0], [math.sin(1.45), 0.0, math.cos(1.45)], [-0.6, 0.2, -0.8], [1.0, 0.0, 0.05]]


def half_envmaps(n, He, We, seed):
    """n fp16 maps [n,He,We,3] on the device, clamped to the fp16 range as a caller would convert them."""
    return torch.stack([synthetic_envmap(He, We, seed=seed + b, device=DEV, as_numpy=False) for b in range(n)]
                       ).clamp(max=65504).half()


@pytest.fixture(scope="module")
def maps_2k():
    return half_envmaps(3, 1000, 2000, 700)


def mixed_inputs(n, n_env, seed):
    """n renders: the mirror Z0, sharp and rough lobes, views from the front, grazing and behind, every other one
    flipped; render k uses envmap k % n_env."""
    rough = [0.0, 0.02, 0.08, 0.15, 0.25, 0.45, 0.8]
    z, view = [], []
    for i in range(n):
        zi = torch.tensor(Z0) if i == 0 else sample_brdf(seed + i)
        if i > 0:
            zi[4] = rough[i % len(rough)]
        z.append(zi)
        view.append(torch.tensor(VIEWS[i % len(VIEWS)]))
    env_index = torch.tensor([i % n_env for i in range(n)], dtype=torch.int32, device=DEV)
    flip = torch.tensor([i % 2 == 1 for i in range(n)], device=DEV)
    return torch.stack(z), torch.stack(view), env_index, flip


def both(env16, *args, **kw):
    """(render of the fp16 maps, render of their fp32 upcast), each checked for a clean status."""
    h = render_batch(env16, *args, check_status=True, **kw).clone()
    f = render_batch(env16.float(), *args, check_status=True, **kw).clone()
    torch.cuda.synchronize()
    return h, f


@pytest.mark.parametrize("S", [1, 2, 4, 8, 16, None])
def test_every_lattice_bit_equal(maps_2k, S):
    z, view, env_index, flip = mixed_inputs(10, 3, 800)
    channel_first = S not in (2, 8)
    h, f = both(maps_2k, z, view, env_index=env_index, flip=flip, res=128, footprint_S=S, channel_first=channel_first)
    assert torch.isfinite(f).all() and f.abs().sum() > 0
    assert torch.equal(h, f)


@pytest.mark.parametrize("He,We,res", [(1000, 2000, 128), (128, 256, 64), (128, 256, 256)])
def test_several_launch_sequences_bit_equal(He, We, res):
    """70 renders over 4 envmaps: two launch sequences of at most 64 renders, auto footprints."""
    env16 = half_envmaps(4, He, We, 900)
    z, view, env_index, flip = mixed_inputs(70, 4, 1000)
    h, f = both(env16, z, view, env_index=env_index, flip=flip, res=res, footprint_S=None)
    assert torch.equal(h, f)


def test_same_traversal(maps_2k):
    """footprint_per_render through the options and collect_stats: the status words (flags, high-water marks, pool
    chunks, cells visited and accepted per pass) are equal, so the tree walk is the same for both texel types."""
    z, view, env_index, flip = mixed_inputs(12, 3, 1100)
    per_render = torch.tensor([1, 2, 4, 8, 16, 0] * 2, dtype=torch.int32, device=DEV)
    status = {}
    outs = {}
    for name, env in (("half", maps_2k), ("float", maps_2k.float())):
        o = _lib.default_render_options()
        o.footprint_per_render = per_render.data_ptr()
        o.collect_stats = 1
        outs[name] = render_batch(env, z, view, env_index=env_index, flip=flip, res=128, footprint_S=None, options=o,
                                  check_status=True).clone()
        status[name] = list(render_batch.last_status)
    assert torch.equal(outs["half"], outs["float"])
    assert status["half"][0:12] == status["float"][0:12]
    assert status["half"][16:36] == status["float"][16:36]
    assert sum(status["half"][16:36]) > 0


def test_drop_in_renderer_keeps_fp16(maps_2k):
    env16 = maps_2k[0]
    z = sample_brdf(1200)
    runs = {}
    for name, env in (("half", env16), ("float", env16.float())):
        r = B200RefMapRenderer(refmap_res=128, brdf_param_names=BRDF_PARAM_NAMES, envmap_size=(1000, 2000))
        a = r.rendering(z, BRDF_PARAM_NAMES, envmap=env, view_from=torch.tensor(VIEWS[1]), flip=True)
        assert r._envmap.dtype == env.dtype
        b = r.rendering(z * 0.5, BRDF_PARAM_NAMES, envmap=None)
        c = r.rendering(z, BRDF_PARAM_NAMES, envmap=env, view_from=torch.tensor(VIEWS[2]), new_scene=True)
        runs[name] = (a, b, c)
    for x, y in zip(runs["half"], runs["float"]):
        assert torch.equal(x, y)


def test_batched_callers_bit_equal(maps_2k):
    B, L = 3, 2
    z = torch.stack([torch.stack([sample_brdf(1300 + 10 * l + b) for b in range(B)]) for l in range(L)])  # [L,B,6]
    views = torch.stack([sample_view(1300 + b) for b in range(B)])
    out = {}
    for name, env in (("half", maps_2k), ("float", maps_2k.float())):
        r = B200RefMapRenderer(refmap_res=64, brdf_param_names=BRDF_PARAM_NAMES, envmap_size=(1000, 2000))
        refmaps = rendering_refmaps(r, env, z, view_from=views)
        assert r._envmap.dtype == env.dtype
        post, scale, raw = synthesize_refmaps(r, z, env, views)
        out[name] = (refmaps, scale, raw, *post)
    for x, y in zip(out["half"], out["float"]):
        assert torch.equal(x, y)


def test_flat_path_upcasts():
    env16 = half_envmaps(2, 64, 128, 1400)
    z, view, env_index, flip = mixed_inputs(2, 2, 1500)
    h = render_batch(env16, z, view, env_index=env_index, flip=flip, res=16, footprint_S=2, flat=True)
    f = render_batch(env16.float(), z, view, env_index=env_index, flip=flip, res=16, footprint_S=2, flat=True)
    assert torch.equal(h, f)


def test_cpu_map_rejected_and_strided_map_read_in_place(maps_2k, monkeypatch):
    z, view, env_index, flip = mixed_inputs(4, 2, 1600)
    with pytest.raises(RuntimeError, match="no CPU path"):
        render_batch(maps_2k[:2].cpu(), z, view, env_index=env_index)
    # a channel-first buffer seen as [B,He,We,3]: not contiguous
    strided = maps_2k[:2].permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)
    assert not strided.is_contiguous() and strided.dtype == torch.float16
    L = _lib.lib()
    calls = []
    half_entry = L.drm_render_refmaps_half

    def counting(*args):
        calls.append(args)
        return half_entry(*args)

    monkeypatch.setattr(L, "drm_render_refmaps_half", counting)
    h = render_batch(strided, z, view, env_index=env_index, flip=flip, res=64, footprint_S=None)
    assert len(calls) == 1
    monkeypatch.undo()
    f = render_batch(maps_2k[:2].float(), z, view, env_index=env_index, flip=flip, res=64, footprint_S=None)
    assert torch.equal(h, f)


def test_abi_entry_validates_like_the_fp32_one(maps_2k):
    """drm_render_refmaps_half rejects what drm_render_refmaps_opts rejects, with the same status."""
    L = _lib.lib()
    ws = torch.empty(64, dtype=torch.uint8, device=DEV)
    z = torch.zeros(1, 6, device=DEV)
    v = torch.tensor([[0.0, 0.0, 1.0]], device=DEV)
    idx = torch.zeros(1, dtype=torch.int32, device=DEV)
    out = torch.empty(1, 3, 16, 16, device=DEV)
    stream = torch.cuda.current_stream().cuda_stream
    for S, nbytes in ((3, ws.numel()), (1, 64)):  # bad footprint; workspace too small
        codes = [fn(maps_2k.data_ptr(), 3, 1000, 2000, idx.data_ptr(), z.data_ptr(), v.data_ptr(), None, 1, 16, S,
                    0.0, 1, out.data_ptr(), ws.data_ptr(), nbytes, stream, ctypes.POINTER(_lib.RenderOptions)())
                 for fn in (L.drm_render_refmaps_half, L.drm_render_refmaps_opts)]
        assert codes[0] == codes[1] != _lib.DRM_OK
