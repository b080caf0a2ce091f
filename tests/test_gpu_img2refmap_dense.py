"""img2refmap_images (drm_img2refmap_dense) against the route it replaces: boolean-mask compaction, offsets and
img2refmap_batch.  Every output is compared with torch.equal; the compacted route's sel_index (a compacted image-local
index) is mapped through the compaction to the dense index y*W + x."""
import numpy as np
import pytest
import torch

from drmnet_b200.img2refmap import img2refmap_batch, img2refmap_images
from drmnet_b200.synth import sphere_normals

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SYNTH = ["A_half_cell_res32", "B_small_window_res64", "C_overlap_res256", "D_min_points_res32", "E_nan_ties_res16",
         "G_nan_angles_res16", "F_wide_window_res24"]


def compacted(colors, normals, mask, res, thr, mp=0, reduce="median", channel_first=False):
    """Today's route on dense tensors, with sel_index mapped to the dense image-local index."""
    if channel_first:
        colors, normals = colors.permute(0, 2, 3, 1), normals.permute(0, 2, 3, 1)
    B, H, W = colors.shape[:3]
    if mask is None:
        mask = torch.ones((B, H, W), dtype=torch.bool, device=colors.device)
    offsets = torch.zeros(B + 1, dtype=torch.int64, device=colors.device)
    offsets[1:] = mask.sum((1, 2)).cumsum(0)
    refmap, refmask, counts, sel = img2refmap_batch(colors[mask], normals[mask], offsets, res, thr, mp, reduce=reduce)
    dense = sel.clone()
    for b in range(B):
        idx = mask[b].flatten().nonzero().squeeze(1).to(torch.int32)  # row-major, the order boolean indexing keeps
        hit = sel[b] >= 0
        dense[b][hit] = idx[sel[b][hit].long()]
    return refmap, refmask, counts, dense


def assert_same(ours, ref):
    for x, y in zip(ours, ref):
        assert x.shape == y.shape and x.dtype == y.dtype
        if x.is_floating_point():
            assert torch.equal(x.isnan(), y.isnan())
            x, y = x.nan_to_num(nan=0.0), y.nan_to_num(nan=0.0)
        assert torch.equal(x, y)


def embed(colors, normals, H, W, seed, fill=float("nan")):
    """n listed pixels placed, in their order, at n random row-major positions of an H x W image; the pixels outside
    the mask hold `fill` (NaN: they must not be read into any output)."""
    n = len(colors)
    rng = np.random.default_rng(seed)
    pos = np.sort(rng.choice(H * W, n, replace=False))
    col = np.full((H * W, colors.shape[1]), fill, np.float32)
    nrm = np.full((H * W, 3), fill, np.float32)
    col[pos], nrm[pos] = colors, normals
    mask = np.zeros(H * W, bool)
    mask[pos] = True
    return col.reshape(H, W, -1), nrm.reshape(H, W, 3), mask.reshape(H, W)


def to_layout(x, channel_first):
    """[B,H,W,C] -> a [B,C,H,W] tensor when channel_first (contiguous in that layout)."""
    return x.permute(0, 3, 1, 2).contiguous() if channel_first else x


def sphere_batch(B, radius, seed, noise=0.05):
    """Dense sphere normal images (sphere_normals, perturbed as normalise(n + N(0, noise)) inside the sphere) with
    smooth HDR-like colours plus noise, [B,2r,2r,3] each, and the ObsNet mask ||n|| > 0.5."""
    n0, m = sphere_normals(radius)
    g = torch.Generator().manual_seed(seed)
    n = torch.from_numpy(n0)[None].repeat(B, 1, 1, 1)
    n = n + noise * torch.randn(n.shape, generator=g)
    n = torch.where(torch.from_numpy(m)[None, ..., None], n / n.norm(dim=-1, keepdim=True), torch.zeros(()))
    col = torch.exp(1.5 * n[..., :1] + 0.7 * n[..., 1:2]) * torch.tensor([1.0, 0.9, 0.8]) \
        + 40.0 * torch.exp(-((n[..., :1] - 0.3) ** 2 + (n[..., 1:2] - 0.5) ** 2) / 0.002)
    col = col * (1 + 0.01 * torch.randn(col.shape, generator=g))
    n, col = n.float().to(DEV), col.float().to(DEV)
    return col, n, n.norm(dim=-1) > 0.5


@pytest.mark.parametrize("channel_first", [False, True])
def test_sample_golden_in_a_256_image(golden_sample, channel_first):
    g = golden_sample
    col, nrm, m = embed(g["colors"], g["normals"], 256, 256, seed=1)
    col, nrm = to_layout(torch.from_numpy(col)[None].to(DEV), channel_first), to_layout(torch.from_numpy(nrm)[None].to(DEV), channel_first)
    mask = torch.from_numpy(m)[None].to(DEV)
    res, thr = 128, float(g["thr"])
    ours = img2refmap_images(col, nrm, mask, res, thr, channel_first=channel_first)
    assert_same(ours, compacted(col, nrm, mask, res, thr, channel_first=channel_first))
    refmap, refmask = ours[0][0].cpu().numpy(), ours[1][0].cpu().numpy()
    # the reference's own outputs on data/sample
    assert np.array_equal(refmask, g["refmask"]) and np.array_equal(refmap, g["refmap"])
    assert int(refmask.sum()) == 7621 and abs(float(refmap.astype(np.float64).sum()) - 2173.994606) < 1e-5


@pytest.mark.parametrize("name", SYNTH)
@pytest.mark.parametrize("channel_first", [False, True])
def test_synthetic_cases_in_dense_images(golden_synth, name, channel_first):
    """Each case in image 1 of three: image 0 is another case's pixels, image 2 has an all-false mask.  Covers NaN
    angles (G), NaN colour sums and ties (E), windows wider than a cell (C, F) and min_points (D)."""
    c, other = golden_synth[name], golden_synth["A_half_cell_res32"]
    res, thr, mp = int(c["res"]), float(c["thr"]), int(c["min_points"])
    H, W = 96, 112
    normals = c["normals"].copy()
    normals[np.isnan(c["thetaphi_torch_cpu"]).any(1)] = np.nan  # G's NaN angles as NaN normals
    imgs = [embed(other["colors"], other["normals"], H, W, seed=2), embed(c["colors"], normals, H, W, seed=3),
            embed(other["colors"][:50], other["normals"][:50], H, W, seed=4)]
    col = to_layout(torch.from_numpy(np.stack([i[0] for i in imgs])).to(DEV), channel_first)
    nrm = to_layout(torch.from_numpy(np.stack([i[1] for i in imgs])).to(DEV), channel_first)
    mask = torch.from_numpy(np.stack([i[2] for i in imgs])).to(DEV)
    mask[2] = False
    for reduce in ("median", "mean"):
        ours = img2refmap_images(col, nrm, mask, res, thr, mp, channel_first=channel_first, reduce=reduce)
        assert_same(ours, compacted(col, nrm, mask, res, thr, mp, reduce=reduce, channel_first=channel_first))
        assert not ours[1][2].any() and int(ours[2][2].sum()) == 0
    if name == "G_nan_angles_res16":
        assert np.isnan(normals).any(1).sum() == 3
    if name == "E_nan_ties_res16":
        assert np.isnan(c["colors"].sum(1)).any()


@pytest.mark.parametrize("res", [32, 128, 256])
@pytest.mark.parametrize("reduce", ["median", "mean"])
def test_sphere_batches_across_resolutions(res, reduce):
    col, nrm, mask = sphere_batch(3, 96, seed=res)
    for cells, mp in ((0.5, 0), (1.5, 3)):  # the reference's half-cell window, and a window wider than a cell
        thr = float(np.pi / res * cells)
        ours = img2refmap_images(col, nrm, mask, res, thr, mp, channel_first=False, reduce=reduce, check_status=True)
        assert img2refmap_images.last_status[0] == 0
        assert_same(ours, compacted(col, nrm, mask, res, thr, mp, reduce=reduce))
        assert ours[1].sum() > 0


def test_strided_views_are_read_in_place():
    """A channel slice of a 4-channel image and a permute without contiguous(): read through their strides."""
    col, nrm, mask = sphere_batch(2, 64, seed=5)
    res, thr = 64, float(np.pi / 128)
    want = img2refmap_images(col, nrm, mask, res, thr, channel_first=False)
    rgba = torch.cat([col, torch.full_like(col[..., :1], float("nan"))], -1)  # alpha is NaN: it must not be read
    sliced = rgba[..., :3]
    assert not sliced.is_contiguous()
    assert_same(img2refmap_images(sliced, nrm, mask, res, thr, channel_first=False), want)
    chw_c, chw_n = col.permute(0, 3, 1, 2), nrm.permute(0, 3, 1, 2)  # [B,C,H,W] views of HWC storage
    assert not chw_c.is_contiguous()
    assert_same(img2refmap_images(chw_c, chw_n, mask, res, thr, channel_first=True), want)
    hwc_c, hwc_n = to_layout(col, True).permute(0, 2, 3, 1), to_layout(nrm, True).permute(0, 2, 3, 1)
    assert not hwc_c.is_contiguous()
    assert_same(img2refmap_images(hwc_c, hwc_n, mask, res, thr, channel_first=False), want)
    # one image without the batch dimension
    single = img2refmap_images(chw_c[1], chw_n[1], mask[1], res, thr, channel_first=True)
    assert_same(single, tuple(o[1] for o in want))


def test_mask_none_is_every_pixel():
    col, nrm, _ = sphere_batch(2, 48, seed=6)
    nrm = torch.nn.functional.normalize(nrm + 0.1, dim=-1)  # every pixel has a normal
    res, thr = 32, float(np.pi / 64)
    ours = img2refmap_images(col, nrm, None, res, thr, channel_first=False)
    assert_same(ours, compacted(col, nrm, None, res, thr))
    full = torch.ones(col.shape[:3], dtype=torch.bool, device=DEV)
    assert_same(ours, img2refmap_images(col, nrm, full, res, thr, channel_first=False))


def test_batches_beyond_the_per_call_pixel_limit_are_split(monkeypatch):
    import drmnet_b200.img2refmap as M
    col, nrm, mask = sphere_batch(5, 32, seed=8)
    mask[3] = False
    res, thr = 32, float(np.pi / 64)
    whole = img2refmap_images(col, nrm, mask, res, thr, channel_first=False)
    monkeypatch.setattr(M, "MAX_PIXELS_PER_CALL", 2 * 64 * 64 + 100)  # two images per call: 3 calls
    calls = []
    real = M._lib.lib()

    class Spy:
        def __getattr__(self, name):
            return getattr(real, name)

        def drm_img2refmap_dense(self, *args):
            calls.append(args[5])
            return real.drm_img2refmap_dense(*args)

    monkeypatch.setattr(M._lib, "lib", lambda spy=Spy(): spy)
    parts = img2refmap_images(col, nrm, mask, res, thr, channel_first=False)
    assert calls == [2, 2, 1]
    assert_same(parts, whole)
    monkeypatch.setattr(M, "MAX_PIXELS_PER_CALL", 64 * 64 - 1)
    with pytest.raises(ValueError, match="one image"):
        img2refmap_images(col, nrm, mask, res, thr, channel_first=False)


def test_run_to_run_determinism():
    col, nrm, mask = sphere_batch(4, 128, seed=9)
    col = torch.round(col * 8) / 8  # many equal channel sums: the order falls back to the pixel index
    outs = [img2refmap_images(col, nrm, mask, 16, float(np.pi / 32), channel_first=False) for _ in range(3)]
    for o in outs[1:]:
        assert_same(o, outs[0])
    assert_same(outs[0], compacted(col, nrm, mask, 16, float(np.pi / 32)))


def test_no_host_synchronisation():
    col, nrm, mask = sphere_batch(2, 64, seed=10)
    img2refmap_images(col, nrm, mask, 64, float(np.pi / 128), channel_first=False)  # loads the library
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = img2refmap_images(col, nrm, mask, 64, float(np.pi / 128), channel_first=False)
        with pytest.raises(RuntimeError):
            compacted(col, nrm, mask, 64, float(np.pi / 128))
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert_same(out, compacted(col, nrm, mask, 64, float(np.pi / 128)))


def test_errors_match_the_batch_entry():
    col, nrm, mask = sphere_batch(1, 16, seed=11)
    with pytest.raises(TypeError):
        img2refmap_images(col.double(), nrm, mask, 16, 0.1, channel_first=False)
    with pytest.raises(TypeError):
        img2refmap_images(col, nrm, mask, 16, None, channel_first=False)
    with pytest.raises(TypeError):
        img2refmap_images(col, nrm, mask.float(), 16, 0.1, channel_first=False)
    with pytest.raises(ValueError):
        img2refmap_images(col, nrm[..., :2], mask, 16, 0.1, channel_first=False)
    with pytest.raises(ValueError):
        img2refmap_images(col, nrm, mask[:, :8], 16, 0.1, channel_first=False)
    with pytest.raises(ValueError, match="C=5"):
        c5 = torch.zeros(1, 32, 32, 5, device=DEV)
        img2refmap_images(c5, nrm, mask, 16, 0.1, channel_first=False)
    with pytest.raises(RuntimeError, match="no CPU path"):
        img2refmap_images(col.cpu(), nrm, mask, 16, 0.1, channel_first=False)


def test_config3_chain_on_dense_images():
    """render -> refmap_lookup on a dense normal image -> img2refmap_images equals the compacted chain of
    tests/test_gpu_callers.py (lookup of the masked normals, then img2refmap_batch)."""
    from drmnet_b200.callers import refmap_lookup
    from drmnet_b200.renderer import render_batch
    from drmnet_b200.synth import synthetic_envmap
    res = 128
    env = torch.from_numpy(synthetic_envmap(250, 500, seed=9)).to(DEV)
    z = torch.tensor([[0.3, 0.8, 0.6, 0.4, 0.5, 0.7]])
    refmap = render_batch(env[None], z, torch.tensor([[0.0, 0.0, 1.0]]), res=res, footprint_S=1)  # [1,3,res,res]
    n, m = sphere_normals(128)
    thr = float(np.pi / res / 2)
    # compacted chain
    normals = torch.from_numpy(n[m]).to(DEV)
    colors = refmap_lookup(refmap, normals)
    offsets = torch.tensor([0, normals.shape[0]], dtype=torch.int64, device=DEV)
    want = img2refmap_batch(colors, normals, offsets, res, thr)
    # dense chain: shade every pixel of the image, scatter under the mask
    dense_n = torch.from_numpy(n).to(DEV)  # [256,256,3], zero outside the sphere
    dense_c = refmap_lookup(refmap, dense_n.view(-1, 3)).view(256, 256, 3)
    mask = dense_n.norm(dim=-1) > 0.5
    assert torch.equal(mask.cpu(), torch.from_numpy(m))
    ours = img2refmap_images(dense_c, dense_n, mask, res, thr, channel_first=False)
    idx = mask.flatten().nonzero().squeeze(1).to(torch.int32)
    sel = torch.where(want[3] >= 0, idx[want[3].clamp_min(0).long()], want[3])
    assert_same((o[None] for o in ours), (*want[:3], sel))
    assert ours[1].sum() > 0.6 * res * res
