"""Envmap banks.  A bank renders with diffuse pyramids built once, by the same kernels and launches the render uses on
the maps it is given, and the render kernels read them at the same offsets.  So every render from a bank must be
bit-identical to ``render_batch`` on the plain maps: every lattice, fp32 and fp16, several launch sequences, sparse
and permuted slots, the drop-in renderer and the training path."""
import math

import pytest
import torch

from drmnet_b200 import _lib
from drmnet_b200.callers import synthesize_refmaps
from drmnet_b200.renderer import B200RefMapRenderer, EnvmapBank, render_batch
from drmnet_b200.synth import BRDF_PARAM_NAMES, Z0, sample_brdf, sample_view, synthetic_envmap

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
VIEWS = [[0.0, 0.0, 1.0], [math.sin(1.45), 0.0, math.cos(1.45)], [-0.6, 0.2, -0.8], [1.0, 0.0, 0.05]]


def envmaps(n, He, We, seed, half=False):
    e = torch.stack([synthetic_envmap(He, We, seed=seed + b, device=DEV, as_numpy=False) for b in range(n)])
    return e.clamp(max=65504).half() if half else e


@pytest.fixture(scope="module")
def maps_2k():
    return envmaps(3, 1000, 2000, 2100)


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


def both(env, *args, **kw):
    """(render from a bank of the maps, render of the plain maps), each checked for a clean status."""
    b = render_batch(EnvmapBank(env), *args, check_status=True, **kw).clone()
    p = render_batch(env, *args, check_status=True, **kw).clone()
    torch.cuda.synchronize()
    return b, p


@pytest.mark.parametrize("S", [1, 2, 4, 8, 16, None])
@pytest.mark.parametrize("half", [False, True])
def test_every_lattice_bit_equal(maps_2k, S, half):
    env = maps_2k.clamp(max=65504).half() if half else maps_2k
    z, view, env_index, flip = mixed_inputs(10, 3, 2200)
    channel_first = S not in (2, 8)
    b, p = both(env, z, view, env_index=env_index, flip=flip, res=128, footprint_S=S, channel_first=channel_first)
    assert torch.isfinite(p).all() and p.abs().sum() > 0
    assert torch.equal(b, p)


@pytest.mark.parametrize("He,We,res", [(1000, 2000, 128), (128, 256, 64), (128, 256, 256)])
@pytest.mark.parametrize("half", [False, True])
def test_several_launch_sequences_bit_equal(He, We, res, half):
    """70 renders over 4 envmaps: two launch sequences of at most 64 renders, auto footprints."""
    env = envmaps(4, He, We, 2300, half)
    z, view, env_index, flip = mixed_inputs(70, 4, 2400)
    b, p = both(env, z, view, env_index=env_index, flip=flip, res=res, footprint_S=None)
    assert torch.equal(b, p)


@pytest.mark.parametrize("half", [False, True])
def test_sparse_permuted_slots_of_a_large_bank(half):
    """A bank of 300 small maps, renders that use 9 of them in a scattered order: equal to the same renders on just
    the 9 maps they use."""
    env = envmaps(300, 128, 256, 2500, half)
    bank = EnvmapBank(env)
    used = [297, 3, 150, 0, 42, 299, 77, 200, 11]
    n = 20
    slots = torch.tensor([used[(5 * i + 2) % len(used)] for i in range(n)], dtype=torch.int32, device=DEV)
    z, view, _, flip = mixed_inputs(n, 1, 2600)
    a = render_batch(bank, z, view, env_index=slots, flip=flip, res=64, footprint_S=None, check_status=True).clone()
    local = torch.tensor([used.index(int(s)) for s in slots], dtype=torch.int32, device=DEV)
    sub = env[torch.tensor(used, device=DEV)]
    c = render_batch(sub, z, view, env_index=local, flip=flip, res=64, footprint_S=None, check_status=True)
    assert torch.equal(a, c)


def test_same_traversal(maps_2k):
    """footprint_per_render and collect_stats: the status words (flags, high-water marks, pool chunks, cells visited
    and accepted per pass) are equal, so the tree walk is the same."""
    z, view, env_index, flip = mixed_inputs(12, 3, 2700)
    per_render = torch.tensor([1, 2, 4, 8, 16, 0] * 2, dtype=torch.int32, device=DEV)
    status, outs = {}, {}
    bank = EnvmapBank(maps_2k)
    for name, env in (("bank", bank), ("plain", maps_2k)):
        o = _lib.default_render_options()
        o.footprint_per_render = per_render.data_ptr()
        o.collect_stats = 1
        outs[name] = render_batch(env, z, view, env_index=env_index, flip=flip, res=128, footprint_S=None, options=o,
                                  check_status=True).clone()
        status[name] = list(render_batch.last_status)
    assert torch.equal(outs["bank"], outs["plain"])
    assert status["bank"][0:12] == status["plain"][0:12]
    assert status["bank"][16:36] == status["plain"][16:36]
    assert sum(status["bank"][16:36]) > 0


@pytest.mark.parametrize("half", [False, True])
def test_update_equals_a_fresh_bank_and_stale_bank_raises(half):
    env = envmaps(6, 128, 256, 2800, half)
    z, view, env_index, flip = mixed_inputs(12, 6, 2900)
    kw = dict(env_index=env_index, flip=flip, res=64, footprint_S=None)
    bank = EnvmapBank(env)
    assert bank.maps.data_ptr() == env.data_ptr()  # contiguous in its storage type: used in place
    # new maps copied into two slots
    new = envmaps(2, 128, 256, 3000, half)
    bank.update([4, 1], new)
    ref = env.clone()
    ref[4], ref[1] = new[0], new[1]
    assert torch.equal(bank.maps, ref)
    assert torch.equal(render_batch(bank, z, view, **kw), render_batch(EnvmapBank(ref.clone()), z, view, **kw))
    # an in-place edit of the caller's tensor: refused until update() re-reads the slot
    env[2] *= 0.25
    assert bank.stale
    with pytest.raises(RuntimeError, match="update"):
        render_batch(bank, z, view, **kw)
    bank.update(torch.tensor([2]))
    assert not bank.stale
    out = render_batch(bank, z, view, **kw)
    assert torch.equal(out, render_batch(env.clone(), z, view, **kw))
    assert torch.equal(out, render_batch(EnvmapBank(env.clone()), z, view, **kw))
    with pytest.raises(IndexError):
        bank.update([6])
    # a converted copy does not follow the caller's tensor, so the caller's edits do not make it stale
    f64 = env.double()
    conv = EnvmapBank(f64)
    f64 *= 2
    assert not conv.stale and conv.maps.dtype == torch.float32


def test_flat_path_renders_the_bank_maps():
    env = envmaps(2, 64, 128, 3100)
    z, view, env_index, flip = mixed_inputs(2, 2, 3200)
    a = render_batch(EnvmapBank(env), z, view, env_index=env_index, flip=flip, res=16, footprint_S=2, flat=True)
    b = render_batch(env, z, view, env_index=env_index, flip=flip, res=16, footprint_S=2, flat=True)
    assert torch.equal(a, b)


def _plain(env, z6, view, flip, res=128, S=None):
    return render_batch(env[None], z6[None], torch.as_tensor(view, dtype=torch.float32)[None].to(DEV),
                        flip=torch.tensor([flip], device=DEV), res=res, footprint_S=S, channel_first=False)[0]


def test_drop_in_renderer_sequence(maps_2k):
    """The get_input loop: an envmap, then None x 3 with new_scene in between, an in-place edit of the persistent
    map, then an fp16 map.  Every image equals render_batch on the same map; after the first call, a call with
    envmap=None launches fewer kernels by exactly the diffuse pyramid build."""
    L = _lib.lib()
    env = maps_2k[0].clone()
    r = B200RefMapRenderer(refmap_res=128, brdf_param_names=BRDF_PARAM_NAMES, envmap_size=(1000, 2000))
    zs = [sample_brdf(3300 + i) for i in range(8)]
    v1, v2 = torch.tensor(VIEWS[1]), torch.tensor(VIEWS[2])

    def z6_of(z):
        return z.float().clip(0, 1).to(DEV)

    img = r.rendering(zs[0], BRDF_PARAM_NAMES, envmap=env, view_from=v1, flip=True)
    assert torch.equal(img, _plain(env, z6_of(zs[0]), v1, True))
    # envmap=None: the bank is reused
    n0 = L.drm_launch_count()
    img = r.rendering(zs[1], BRDF_PARAM_NAMES)
    n_bank = L.drm_launch_count() - n0
    assert torch.equal(img, _plain(env, z6_of(zs[1]), v1, True))
    n0 = L.drm_launch_count()
    _plain(env, z6_of(zs[1]), v1, True)
    n_plain = L.drm_launch_count() - n0
    n0 = L.drm_launch_count()
    EnvmapBank(env[None])
    n_build = L.drm_launch_count() - n0
    # the build's launches, less its direction tables (which every render computes for itself)
    assert n_build - 1 >= 2 and n_plain - n_bank == n_build - 1
    # new_scene renders with its own envmap and leaves the persistent one alone
    other = maps_2k[1]
    img = r.rendering(zs[2], BRDF_PARAM_NAMES, envmap=other, view_from=v2, new_scene=True)
    assert torch.equal(img, _plain(other, z6_of(zs[2]), v2, False))
    img = r.rendering(zs[3], BRDF_PARAM_NAMES)
    assert torch.equal(img, _plain(env, z6_of(zs[3]), v1, True))
    # an in-place edit of the persistent map is seen, as before banks
    env[100:300] *= 3.0
    img = r.rendering(zs[4], BRDF_PARAM_NAMES)
    assert torch.equal(img, _plain(env, z6_of(zs[4]), v1, True))
    img = r.rendering(zs[5], BRDF_PARAM_NAMES, view_from=v2, flip=False)
    assert torch.equal(img, _plain(env, z6_of(zs[5]), v2, False))
    # an fp16 map stays fp16
    env16 = maps_2k[2].clamp(max=65504).half()
    img = r.rendering(zs[6], BRDF_PARAM_NAMES, envmap=env16)
    assert r._envmap.dtype == torch.float16
    assert torch.equal(img, _plain(env16, z6_of(zs[6]), v2, False))
    img = r.rendering(zs[7], BRDF_PARAM_NAMES)
    assert torch.equal(img, _plain(env16, z6_of(zs[7]), v2, False))


@pytest.mark.parametrize("half", [False, True])
def test_synthesize_refmaps_from_a_bank(half):
    """The training path: batch element b uses bank slot env_ids[b]; equal to the same call on the gathered maps,
    cache misses included."""
    env = envmaps(40, 1000, 2000, 3400, half) if half else envmaps(40, 128, 256, 3400)
    bank = EnvmapBank(env)
    B, G = 6, 3
    env_ids = torch.tensor([39, 5, 5, 0, 17, 22], device=DEV)
    z = torch.stack([torch.stack([sample_brdf(3500 + 10 * g + b) for b in range(B)]) for g in range(G)])
    views = torch.stack([sample_view(3500 + b) for b in range(B)])
    r = B200RefMapRenderer(refmap_res=64, brdf_param_names=BRDF_PARAM_NAMES, envmap_size=tuple(env.shape[1:3]))
    cached = [None, torch.full((B, 3, 64, 64), float("nan"), device=DEV), None]
    cached[1][1] = 1.0  # one hit
    a = synthesize_refmaps(r, z, bank, views, cached=cached, env_ids=env_ids)
    b = synthesize_refmaps(r, z, env[env_ids], views, cached=cached)
    for x, y in zip((*a[0], a[1], a[2]), (*b[0], b[1], b[2])):
        assert torch.equal(x, y)
