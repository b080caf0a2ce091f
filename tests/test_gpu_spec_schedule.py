"""The specular passes hand their (render, tile) items to persistent CTAs in a run-time order (a work counter, rim tiles
first).  Whatever CTA takes an item and whenever, every refmap cell must come out bit-identical: across repeated calls
and whether a render shares its call with others or not."""
import math

import pytest
import torch

from drmnet_b200.renderer import render_batch
from drmnet_b200.synth import sample_brdf, synthetic_envmap

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def mixed_batch():
    """20 renders of 3 envmaps at 2000 x 1000: every footprint 1..16 (four S = 16), sharp and rough lobes, views from
    the front, grazing and from behind (the refmap's rim band is where the traversal is longest)."""
    envs = torch.stack([synthetic_envmap(1000, 2000, seed=300 + b, device=DEV, as_numpy=False) for b in range(3)])
    S = [1, 2, 4, 8, 16] * 4
    rough = {1: 0.8, 2: 0.45, 4: 0.25, 8: 0.15, 16: 0.02}
    views = [[0.0, 0.0, 1.0], [math.sin(1.45), 0.0, math.cos(1.45)], [-0.6, 0.2, -0.8], [1.0, 0.0, 0.05]]
    z, view = [], []
    for i, s in enumerate(S):
        zi = sample_brdf(500 + i)
        zi[4] = rough[s]
        z.append(zi)
        view.append(torch.tensor(views[(i // 5 + i) % len(views)]))
    env_index = torch.tensor([i % 3 for i in range(len(S))], dtype=torch.int32)
    return envs, torch.stack(z), torch.stack(view), env_index, S


def _render(envs, z, view, env_index, S):
    out = render_batch(envs, z, view, env_index=env_index.to(DEV), res=128, footprint_S=S, check_status=True)
    torch.cuda.synchronize()
    return out.clone()


def test_repeated_calls_bit_equal(mixed_batch):
    first = _render(*mixed_batch)
    for _ in range(2):
        assert torch.equal(_render(*mixed_batch), first)


def test_split_calls_bit_equal(mixed_batch):
    envs, z, view, env_index, S = mixed_batch
    whole = _render(*mixed_batch)
    for lo, hi in [(0, 7), (7, 8), (8, 20)]:
        part = _render(envs, z[lo:hi], view[lo:hi], env_index[lo:hi], S[lo:hi])
        assert torch.equal(part, whole[lo:hi]), (lo, hi)
