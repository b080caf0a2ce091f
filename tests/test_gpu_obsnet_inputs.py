"""Dense refmap lookup and ObsNet's inputs in one call (GPU): ``refmap_lookup_images`` against compaction followed by
``refmap_lookup``, ``obsnet_inputs`` against the same steps taken call by call, no host synchronisation, and
``rendering_refmaps`` on an envmap bank."""
import numpy as np
import pytest
import torch

from drmnet_b200.callers import (normalized_log_apply, obsnet_condition, obsnet_inputs, refmap_lookup,
                                 refmap_lookup_images, rendering_refmaps)
from drmnet_b200.img2refmap import refmap_mask_make
from drmnet_b200.renderer import B200RefMapRenderer, EnvmapBank, render_batch
from drmnet_b200.synth import BRDF_PARAM_NAMES, sphere_normals, synthetic_envmap

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def normal_maps(B, radius, seed):
    """B perturbed sphere normal maps [B,2r,2r,3] (zero outside the sphere) and their mask ||n|| > 0.5."""
    n0, m0 = sphere_normals(radius)
    g = torch.Generator(device=DEV).manual_seed(seed)
    n = torch.from_numpy(n0).to(DEV)[None].repeat(B, 1, 1, 1)
    n = n + 0.05 * torch.randn(n.shape, generator=g, device=DEV)
    inside = torch.from_numpy(m0).to(DEV)[None, ..., None]
    n = torch.where(inside, n / n.norm(dim=-1, keepdim=True), torch.zeros((), device=DEV)).contiguous()
    return n, n.norm(dim=-1) > 0.5


def compacted_image(refmap, nrm_hwc, mask):
    """The route without the dense entry: boolean-mask compaction, refmap_lookup, scatter into a zero image [B,H,W,C]."""
    B, H, W, _ = nrm_hwc.shape
    if mask is None:
        mask = torch.ones((B, H, W), dtype=torch.bool, device=DEV)
    offsets = torch.zeros(B + 1, dtype=torch.int64, device=DEV)
    offsets[1:] = mask.sum((1, 2)).cumsum(0)
    colors = refmap_lookup(refmap, nrm_hwc[mask], offsets)
    img = torch.zeros((B, H, W, refmap.shape[1]), device=DEV)
    img[mask] = colors
    return img


def test_lookup_images_equals_compacted_lookup():
    g = torch.Generator(device=DEV).manual_seed(3)
    nrm, mask = normal_maps(3, 32, seed=1)
    mask[1] = False  # an image with an empty mask
    for C in (3, 1, 4):
        refmap = torch.exp(torch.randn(3, C, 48, 40, generator=g, device=DEV))
        want = compacted_image(refmap, nrm, mask)
        assert torch.equal(refmap_lookup_images(refmap, nrm, mask, channel_first=False), want)
        chw = nrm.permute(0, 3, 1, 2).contiguous()
        assert torch.equal(refmap_lookup_images(refmap, chw, mask, channel_first=True), want.permute(0, 3, 1, 2))
        # a permuted view of the [B,H,W,3] tensor, read through its strides
        assert torch.equal(refmap_lookup_images(refmap, nrm.permute(0, 3, 1, 2), mask, channel_first=True),
                           want.permute(0, 3, 1, 2))
    # a sliced view: a crop of a wider map with spare channels
    big = torch.randn(3, 80, 90, 5, generator=g, device=DEV)
    big[:, 7:71, 11:75, 1:4] = nrm
    view = big[:, 7:71, 11:75, 1:4]
    assert not view.is_contiguous()
    assert torch.equal(refmap_lookup_images(refmap, view, mask, channel_first=False), want)
    # no mask: every pixel, the zero normals outside the sphere included
    assert torch.equal(refmap_lookup_images(refmap, nrm, None, channel_first=False), compacted_image(refmap, nrm, None))


def test_lookup_images_matches_the_reference_refimg(golden_mirmap):
    n, mask = sphere_normals(24)
    refmap = torch.from_numpy(golden_mirmap["refimg_refmap"]).to(DEV)[None]
    nrm = torch.from_numpy(n).to(DEV)[None]  # [1,48,48,3]
    m = torch.from_numpy(mask).to(DEV)[None]
    ours = refmap_lookup_images(refmap, nrm, m, channel_first=False)[0].permute(2, 0, 1).cpu().numpy()
    ref = golden_mirmap["refimg_image"]  # the reference's refmap2refimg_torch
    assert np.abs(ours[:, mask] - ref[:, mask]).max() <= 3e-5 * np.abs(ref[:, mask]).max()
    assert not ours[:, ~mask].any()


def test_lookup_images_argument_errors():
    nrm, mask = normal_maps(2, 8, seed=2)
    refmap = torch.rand(2, 3, 16, 16, device=DEV)
    with pytest.raises(TypeError):
        refmap_lookup_images(refmap, nrm.double(), mask, channel_first=False)
    with pytest.raises(TypeError):
        refmap_lookup_images(refmap, nrm, mask.float(), channel_first=False)
    with pytest.raises(ValueError):
        refmap_lookup_images(refmap[:1], nrm, mask, channel_first=False)
    with pytest.raises(ValueError):
        refmap_lookup_images(refmap, nrm, mask[:, :8], channel_first=False)
    with pytest.raises(ValueError, match="C=5"):
        refmap_lookup_images(torch.rand(2, 5, 16, 16, device=DEV), nrm, mask, channel_first=False)


RES, THR = 32, float(np.pi / 32 / 2)


def scene(B, seed):
    envs = torch.stack([synthetic_envmap(64, 128, seed + b, device=DEV, as_numpy=False) for b in range(B)])
    g = torch.Generator(device=DEV).manual_seed(seed)
    zK = torch.rand(B, 6, generator=g, device=DEV)
    phi = torch.rand(B, generator=g, device=DEV) * 2 * np.pi
    views = torch.stack([torch.sin(phi), torch.zeros_like(phi), torch.cos(phi)], -1)
    nrm, mask = normal_maps(B, 24, seed=seed)
    return envs, zK, views, nrm, mask


def stitched(renderer, envs, zK, views, nrm, mask, **cond_kw):
    """ObsNet's inputs call by call, the way a caller builds them without obsnet_inputs: per image compaction,
    refmap_lookup and refmap_mask_make."""
    LrK = render_batch(envs, zK, views, brdf_param_names=renderer.brdf_param_names, res=RES,
                       footprint_S=renderer.footprint_S, channel_first=True)
    image = torch.zeros((nrm.shape[0], nrm.shape[1], nrm.shape[2], 3), device=DEV)
    maps, masks = [], []
    for b in range(nrm.shape[0]):
        n = nrm[b][mask[b]]
        colors = refmap_lookup(LrK[b], n)
        image[b][mask[b]] = colors
        rm, rk = refmap_mask_make(colors, n, RES, THR)
        maps.append(rm)
        masks.append(rk)
    raw, raw_mask = torch.stack(maps).permute(0, 3, 1, 2).contiguous(), torch.stack(masks)
    cond, cmask, params = obsnet_condition(raw, raw_mask, **cond_kw)
    return cond, cmask, normalized_log_apply(LrK, params), params, raw, raw_mask, image.permute(0, 3, 1, 2)


def assert_same(got, want):
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        if isinstance(a, tuple):
            assert_same(a, b)
        else:
            assert a.shape == b.shape and torch.equal(a, b), f"output {i} differs"


@pytest.mark.parametrize("maps", ["fp32", "fp16", "bank"])
def test_obsnet_inputs_equal_the_stitched_route(maps):
    renderer = B200RefMapRenderer(RES, brdf_param_names=BRDF_PARAM_NAMES)
    envs, zK, views, nrm, mask = scene(3, seed=20)
    chw = nrm.permute(0, 3, 1, 2)
    kw = dict(noisy_observe=0.05, padding_mode="noise", observe_noise=torch.randn(3, 3, RES, RES, device=DEV),
              padding_noise=torch.randn(3, 3, RES, RES, device=DEV))
    if maps == "bank":
        ids = torch.tensor([2, 0, 1], device=DEV)
        got = obsnet_inputs(renderer, zK, EnvmapBank(envs), views, chw, mask, env_ids=ids, angle_threshold=THR, **kw)
        want = stitched(renderer, envs[ids], zK, views, nrm, mask, **kw)
    else:
        e = envs.half() if maps == "fp16" else envs
        got = obsnet_inputs(renderer, zK, e, views, chw, mask, angle_threshold=THR, **kw)
        want = stitched(renderer, e, zK, views, nrm, mask, **kw)
    assert_same(got, want)
    cond, cmask, _, _, _, raw_mask, image = got
    assert cond.shape == (3, 3, RES, RES) and cmask.shape == (3, 1, RES, RES) and image.shape == (3, 3, 48, 48)
    assert raw_mask.dtype == torch.bool and 0.3 * RES * RES < int(raw_mask[0].sum()) < RES * RES
    # the training path: no noise
    assert_same(obsnet_inputs(renderer, zK, envs, views, chw, mask, angle_threshold=THR),
                stitched(renderer, envs, zK, views, nrm, mask))


def test_obsnet_inputs_do_not_synchronise():
    renderer = B200RefMapRenderer(RES, brdf_param_names=BRDF_PARAM_NAMES)
    envs, zK, views, nrm, mask = scene(2, seed=30)
    bank, ids = EnvmapBank(envs), torch.tensor([1, 0], device=DEV)
    chw = nrm.permute(0, 3, 1, 2)
    want = [obsnet_inputs(renderer, zK, envs, views, chw, mask, angle_threshold=THR),  # loads the library, warms up
            obsnet_inputs(renderer, zK, bank, views, chw, mask, env_ids=ids, angle_threshold=THR)]
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = [obsnet_inputs(renderer, zK, envs, views, chw, mask, angle_threshold=THR),
               obsnet_inputs(renderer, zK, bank, views, chw, mask, env_ids=ids, angle_threshold=THR)]
        obsnet_inputs(renderer, zK, bank, views, chw, mask, env_ids=ids, noisy_observe=0.1, padding_mode="noise")
        with pytest.raises(RuntimeError):
            nrm[mask]  # the compaction the dense path does without
    finally:
        torch.cuda.set_sync_debug_mode(0)
    for g, w in zip(got, want):
        assert_same(g, w)


def test_rendering_refmaps_on_a_bank():
    envs, _, views, _, _ = scene(3, seed=40)
    g = torch.Generator(device=DEV).manual_seed(41)
    z = torch.rand(2, 3, 6, generator=g, device=DEV)  # [L,B,P]
    ids = torch.tensor([2, 2, 0], device=DEV)
    bank = EnvmapBank(envs)
    r_bank = B200RefMapRenderer(RES, brdf_param_names=BRDF_PARAM_NAMES)
    r_maps = B200RefMapRenderer(RES, brdf_param_names=BRDF_PARAM_NAMES)
    got = rendering_refmaps(r_bank, bank, z, view_from=views, env_ids=ids)
    want = rendering_refmaps(r_maps, bank.maps[ids], z, view_from=views)
    assert got.shape == (2, 3, 3, RES, RES) and torch.equal(got, want)
    # the stateful renderer ends up holding the same last envmap, view and BRDF vector
    assert torch.equal(r_bank._envmap, r_maps._envmap) and torch.equal(r_bank._envmap, envs[0])
    assert torch.equal(r_bank._view, r_maps._view) and torch.equal(r_bank._bsdf, r_maps._bsdf)
    with pytest.raises(ValueError):
        rendering_refmaps(r_bank, bank, z, view_from=views, env_ids=ids[:2])
