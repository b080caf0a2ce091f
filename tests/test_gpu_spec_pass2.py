"""The default specular pass instances (tree_spec_pass2_kernel<P>) evaluate the sums of the pinned ones
(DrmRenderOptions::spec_kernels = 1) with reordered arithmetic: per refmap the two agree to rounding, on the bench's
renders and on a batch with every footprint, sharp and rough lobes and grazing views.  The fp16 instances give the fp32
result of the upcast map exactly."""
import pytest
import torch

import bench
from drmnet_b200 import _lib
from drmnet_b200.renderer import render_batch
from test_gpu_spec_schedule import mixed_batch  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def options(spec_kernels):
    o = _lib.default_render_options()
    o.spec_kernels = spec_kernels
    return o


def check_close(new, old):
    diff = (new - old).flatten(1).double()
    ref = old.flatten(1).double()
    rel = diff.norm(dim=1) / ref.norm(dim=1)
    worst = diff.abs().amax(dim=1) / ref.abs().amax(dim=1)
    assert rel.max().item() <= 1e-6, f"relative L2 per refmap up to {rel.max().item():.3g}"
    assert worst.max().item() <= 1e-5, f"worst cell up to {worst.max().item():.3g} of the refmap's peak"


def test_bench_renders_match_pinned():
    from drmnet_b200.synth import sample_brdf, sample_view, synthetic_envmap
    envs = torch.stack([synthetic_envmap(bench.HE, bench.WE, seed=1000 + b, device=DEV, as_numpy=False)
                        for b in range(64)])
    z = torch.stack([sample_brdf(1000 + b) for b in range(64)])
    view = torch.stack([sample_view(1000 + b) for b in range(64)])
    S = bench.footprints(z, "auto")
    kw = dict(res=bench.RES, footprint_S=S, check_status=True)
    new = render_batch(envs, z.to(DEV), view.to(DEV), options=options(0), **kw)
    old = render_batch(envs, z.to(DEV), view.to(DEV), options=options(1), **kw)
    check_close(new, old)
    half = render_batch(envs.half(), z.to(DEV), view.to(DEV), options=options(0), **kw)
    up = render_batch(envs.half().float(), z.to(DEV), view.to(DEV), options=options(0), **kw)
    assert torch.equal(half, up)


def test_mixed_batch_matches_pinned(mixed_batch):  # noqa: F811
    envs, z, view, env_index, S = mixed_batch
    kw = dict(env_index=env_index.to(DEV), res=128, footprint_S=S, check_status=True)
    new = render_batch(envs, z, view, options=options(0), **kw)
    old = render_batch(envs, z, view, options=options(1), **kw)
    check_close(new, old)
    half = render_batch(envs.half(), z, view, options=options(0), **kw)
    up = render_batch(envs.half().float(), z, view, options=options(0), **kw)
    assert torch.equal(half, up)


def test_tiny_alpha_min_matches_pinned(mixed_batch):  # noqa: F811
    # lobes far sharper than any default clamp: the reordered loops stay within rounding of the pinned ones
    envs, z, view, env_index, S = mixed_batch
    kw = dict(env_index=env_index.to(DEV), res=128, footprint_S=S, alpha_min=5e-5, check_status=True)
    check_close(render_batch(envs, z, view, options=options(0), **kw), render_batch(envs, z, view, options=options(1), **kw))
