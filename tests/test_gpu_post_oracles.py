"""The kernels around the render against their fp64 oracles (oracle/callers_oracle.py, oracle/img2refmap_oracle.py):
refmap_postprocess, the normalized-log family, mirmap2envmap, both refmap lookups and both img2refmap entries, at the
shapes, channel counts, non-finite inputs and size limits where such kernels go wrong.

Non-finite values follow the reference: NaN must appear exactly where the oracle has NaN, infinities must match with
their sign, and the finite entries are held to the bounds the rest of the suite uses for these kernels."""
import numpy as np
import pytest
import torch

from drmnet_b200 import _lib
from drmnet_b200.callers import (mirmap2envmap, normalized_log_apply, normalized_log_rescale, normalized_log_transform,
                                 obsnet_condition, r0toenvmap, refmap_lookup, refmap_lookup_images, refmap_postprocess)
from drmnet_b200.img2refmap import img2refmap_batch, img2refmap_images, normals_to_thetaphi
from drmnet_b200.synth import sphere_normals
from oracle.callers_oracle import (mirmap2envmap_oracle, normalized_log_apply_oracle, normalized_log_oracle,
                                   normalized_log_rescale_oracle, obsnet_condition_oracle, postprocess_oracle,
                                   refmap_lookup_oracle)
from oracle.img2refmap_oracle import img2refmap_batch_oracle, img2refmap_oracle

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]  # numpy on NaN / inf
DEV = "cuda:0"
INF, NAN = float("inf"), float("nan")


def assert_matches(ours, ref, atol=0.0, rtol=0.0):
    """NaN exactly where ref has NaN, the same infinities, and |ours - ref| <= atol + rtol |ref| elsewhere."""
    ours = ours.detach().cpu().double().numpy() if isinstance(ours, torch.Tensor) else np.asarray(ours, np.float64)
    ref = np.asarray(ref, np.float64)
    assert ours.shape == ref.shape, (ours.shape, ref.shape)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(ours), nan), (f"{int(np.isnan(ours).sum())} NaN, the oracle has {int(nan.sum())}; "
                                                 f"first differing index {np.argwhere(np.isnan(ours) != nan)[0]}")
    inf = np.isinf(ref)
    assert np.array_equal(ours[inf], ref[inf]) and np.isfinite(ours[~nan & ~inf]).all()
    fin = np.isfinite(ref)
    if fin.any():
        excess = np.abs(ours[fin] - ref[fin]) - (atol + rtol * np.abs(ref[fin]))
        assert excess.max() <= 0, f"max |ours - ref| exceeds the bound by {excess.max():.3g}"


def bits(t):
    return t.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ refmap_postprocess

def lrk_stacks(G, N, res, seed):
    """exp(N(0,1)) stacks; LrK holds zero-luminance cells (about 20%) and a few negative-luminance ones.  The negative
    channel value is -1000, so that log10(v * scale + 0.1) is NaN on both sides instead of ill-conditioned near 0."""
    g = torch.Generator().manual_seed(seed)
    x = torch.exp(torch.randn(G, N, 3, res, res, generator=g))
    x[0] *= (torch.rand(N, 1, res, res, generator=g) > 0.2)
    neg = torch.rand(N, res, res, generator=g) < 0.02
    x[0, :, 1][neg] = -1000.0  # L < 0: excluded from the mean like L == 0
    return x


POST_CASES = [(res, G, N) for res in (1, 7, 24, 100, 128, 256, 512) for G, N in ((1, 1), (4, 3), (1, 300), (4, 300))
              if G * N * res * res <= 2e7]


@pytest.mark.parametrize("res,G,N", POST_CASES)
def test_postprocess_shapes(res, G, N):
    """The scale is a mean of fp32 logs over up to 512^2 cells, accumulated by 256 threads in fixed order: rounding
    adds at most ~1e-7 |mean log| per term on average, far below rtol 2e-6 of the scale at every size here."""
    x = lrk_stacks(G, N, res, seed=res * 1000 + N)
    if N >= 3:
        x[0, 1] = 0.0  # all-zero LrK: the mean is 0/0, the scale and the whole sample NaN
    out, scale = refmap_postprocess(x.to(DEV))
    ref, s = postprocess_oracle(x.numpy())
    assert_matches(scale, s, rtol=2e-6)
    assert_matches(out, ref, atol=2e-6)
    if N >= 3:
        assert torch.isnan(scale[1]) and torch.isfinite(scale[0])


@pytest.mark.parametrize("scaler,transform", [(None, "log"), (0.12, None), (None, None), (0.5, "log")])
def test_postprocess_options(scaler, transform):
    """Without the log transform the output is x * scale, one more rounding on the scale's relative error."""
    x = lrk_stacks(3, 5, 24, seed=3)
    out, scale = refmap_postprocess(x.to(DEV), scaler, transform)
    ref, s = postprocess_oracle(x.numpy(), target=scaler, transform=transform)
    assert_matches(scale, s, rtol=2e-6)
    assert_matches(out, ref, **(dict(atol=2e-6) if transform else dict(rtol=2e-6 + 2.0 ** -24)))
    if scaler is None and transform is None:
        assert torch.equal(out.cpu(), x) and torch.all(scale == 1)


def test_postprocess_nonfinite_lrk():
    """NaN luminance makes the sample's scale NaN (log(clip(L)) * (L > 0) is NaN * 0 in the reference); +inf makes it
    0; -inf is L < 0 and excluded; a NaN outside LrK stays in its element.  The finite sample stays exact."""
    x = lrk_stacks(3, 6, 24, seed=4)
    x[0, 1, 1, 5, 7] = NAN
    x[0, 2, 0, 3, 3] = INF
    x[0, 3, 2, 9, 1] = -INF
    x[2, 4, 0, 0, 0] = NAN
    x[0, 5, 0, 2, 2], x[0, 5, 1, 2, 2] = INF, -INF  # L = inf - inf = NaN
    out, scale = refmap_postprocess(x.to(DEV))
    ref, s = postprocess_oracle(x.numpy())
    assert np.isnan(s[1]) and s[2] == 0 and np.isfinite(s[3]) and np.isnan(s[5])
    assert_matches(scale, s, rtol=2e-6)
    assert_matches(out, ref, atol=2e-6)


@pytest.mark.parametrize("res,G,N", [(7, 1, 1), (128, 4, 3), (512, 4, 3), (24, 2, 300)])
def test_postprocess_in_place_through_the_c_abi(res, G, N):
    """include/drmrender.h: in may equal out.  In place equals out of place bit for bit, NaN samples included."""
    x = lrk_stacks(G, N, res, seed=7).to(DEV)
    if N >= 3:
        x[0, 1] = 0.0
    want, want_scale = refmap_postprocess(x)
    buf = x.clone()
    scale = torch.empty(N, device=DEV)
    with torch.cuda.device(DEV):
        _lib.check(_lib.lib().drm_refmap_postprocess(buf.data_ptr(), G, N, res, 0.12, 1, scale.data_ptr(),
                                                     buf.data_ptr(), torch.cuda.current_stream().cuda_stream))
    assert torch.equal(bits(buf), bits(want)) and torch.equal(bits(scale), bits(want_scale))


# ------------------------------------------------------------------------------------------------ normalized-log family

NLOG_SHAPES = [(1, 1), (24, 40), (128, 128), (512, 512)]


def nlog_batch(C, H, W, seed):
    """Five samples with masks: all ones, random, a single cell, empty, random.  Values below the lower bound and
    exact zeros throughout; the single cell's channel 0 is 0, so its minimum is the lower bound exactly."""
    g = torch.Generator().manual_seed(seed)
    x = torch.exp(2 * torch.randn(5, C, H, W, generator=g))
    x *= (torch.rand(5, C, H, W, generator=g) > 0.05)
    x[torch.rand(5, C, H, W, generator=g) < 0.05] = 3e-7  # below lb = 1e-6
    mask = torch.rand(5, H, W, generator=g) > 0.4
    mask[0], mask[2], mask[3] = True, False, False
    mask[2, H // 2, W // 3] = True
    x[2, 0, H // 2, W // 3] = 0.0
    return x, mask


def nlog_params(x, mask):
    _, a, b = normalized_log_oracle(x.numpy(), mask.numpy())
    return a.astype(np.float32), b.astype(np.float32)


@pytest.mark.parametrize("C", [1, 2, 3, 4])
@pytest.mark.parametrize("H,W", NLOG_SHAPES)
def test_normalized_log_family_shapes(C, H, W):
    """The parameters are a log10 of one selected element (no sums), so the bounds do not depend on the size."""
    x, mask = nlog_batch(C, H, W, seed=C * 100 + H)
    out, (lmin, lmax) = normalized_log_transform(x.to(DEV), mask.to(DEV))
    ref, rmin, rmax = normalized_log_oracle(x.numpy(), mask.numpy())
    assert np.isneginf(rmax[3]) and np.isnan(ref[3]).all()  # empty mask: log10(0) parameters, NaN output
    assert_matches(lmin, rmin, atol=2e-6)
    assert_matches(lmax, rmax, atol=2e-6)
    assert_matches(out, ref, atol=2e-5)
    # cond, plain and with both noises
    cond, m, (cmin, cmax) = obsnet_condition(x.to(DEV), mask.to(DEV))
    rc, _, _ = obsnet_condition_oracle(x.numpy(), mask.numpy())
    assert_matches(cond, rc, atol=2e-5)
    assert torch.equal(bits(cmin), bits(lmin)) and torch.equal(bits(cmax), bits(lmax))
    g = torch.Generator().manual_seed(C)
    n1, n2 = torch.randn(x.shape, generator=g), torch.randn(x.shape, generator=g)
    cond, _, _ = obsnet_condition(x.to(DEV), mask.to(DEV), noisy_observe=0.1, observe_noise=n1, padding_mode="noise",
                                  padding_noise=n2)
    rc, _, _ = obsnet_condition_oracle(x.numpy(), mask.numpy(), noisy_observe=0.1, observe_noise=n1.numpy(),
                                       padding_noise=n2.numpy())
    assert_matches(cond, rc, atol=2e-5)
    # fixed parameters (the oracle's, in fp32, given to both sides) and the way back.  Where max == min (one value under
    # the mask) x / 0 is +-inf or NaN by the last bit of log10(x), so such samples get a range of one decade instead
    a, b = nlog_params(x, mask)
    b[a == b] += 1
    p = (torch.from_numpy(a), torch.from_numpy(b))
    t = normalized_log_apply(x.to(DEV), p)
    rt = normalized_log_apply_oracle(x.numpy(), a, b)
    assert_matches(t, rt, atol=2e-5)
    y = torch.clamp(torch.from_numpy(np.nan_to_num(rt, nan=0.0, posinf=0.0, neginf=0.0)).float(), -1.5, 1.5)
    for clamp in (0.0, 0.5):
        back = normalized_log_rescale(y.to(DEV), p, clamp)
        assert_matches(back, normalized_log_rescale_oracle(y.numpy(), a, b, clamp), rtol=3e-5)


def nonfinite_batch(C=3, H=24, W=40):
    """Six samples under random masks: finite, +inf in a masked cell, +inf in an unmasked cell (inf * 0), NaN in a
    masked cell, NaN in an unmasked cell, finite.  Every non-finite sample is NaN in the reference."""
    g = torch.Generator().manual_seed(21)
    x = torch.exp(2 * torch.randn(6, C, H, W, generator=g))
    x[:, :, :3] = 0.0
    mask = torch.rand(6, H, W, generator=g) > 0.4
    mask[:, 5, 6], mask[:, 7, 8] = True, False
    x[1, C - 1, 5, 6] = INF
    x[2, 0, 7, 8] = INF
    x[3, 0, 5, 6] = NAN
    x[4, C - 1, 7, 8] = NAN
    return x, mask


def test_normalized_log_nonfinite_inputs():
    x, mask = nonfinite_batch()
    out, (lmin, lmax) = normalized_log_transform(x.to(DEV), mask.to(DEV))
    ref, rmin, rmax = normalized_log_oracle(x.numpy(), mask.numpy())
    assert np.isfinite(rmin[[0, 5]]).all() and np.isnan(rmin[1:5]).all() and np.isnan(ref[1:5]).all()
    assert_matches(lmin, rmin, atol=2e-6)
    assert_matches(lmax, rmax, atol=2e-6)
    assert_matches(out, ref, atol=2e-5)


@pytest.mark.parametrize("noise", [False, True])
def test_obsnet_condition_nonfinite_inputs(noise):
    x, mask = nonfinite_batch()
    kw, okw = {}, {}
    if noise:
        g = torch.Generator().manual_seed(22)
        n1, n2 = torch.randn(x.shape, generator=g), torch.randn(x.shape, generator=g)
        kw = dict(noisy_observe=0.1, observe_noise=n1, padding_mode="noise", padding_noise=n2)
        okw = dict(noisy_observe=0.1, observe_noise=n1.numpy(), padding_noise=n2.numpy())
    cond, _, (lmin, lmax) = obsnet_condition(x.to(DEV), mask.to(DEV), **kw)
    ref, rmin, rmax = obsnet_condition_oracle(x.numpy(), mask.numpy(), **okw)
    assert np.isnan(ref[1:5]).all()
    assert_matches(lmin, rmin, atol=2e-6)
    assert_matches(lmax, rmax, atol=2e-6)
    assert_matches(cond, ref, atol=2e-5)


def test_normalized_log_apply_and_rescale_nonfinite_inputs():
    """Element-wise: NaN stays NaN both ways (clip and clamp keep it), +inf maps to +inf or to 10^clamp, -inf to the
    lower bound or to 0."""
    x, mask = nonfinite_batch()
    a, b = nlog_params(x[[0, 5]], mask[[0, 5]])
    a, b = np.resize(a, 6), np.resize(b, 6)
    p = (torch.from_numpy(a), torch.from_numpy(b))
    x[0, 1, 4, 4], x[0, 1, 4, 5] = -INF, NAN
    t = normalized_log_apply(x.to(DEV), p)
    rt = normalized_log_apply_oracle(x.numpy(), a, b)
    assert np.isnan(rt).sum() == 3 and np.isposinf(rt).sum() == 2
    assert_matches(t, rt, atol=2e-5)
    y = torch.from_numpy(np.nan_to_num(rt, nan=0.0, posinf=1.0, neginf=-1.0)).float()
    y[0, 0, 10, 10], y[1, 1, 10, 11], y[2, 2, 11, 11], y[3, 0, 12, 12] = NAN, INF, -INF, 1.5
    for clamp in (0.0, 0.5):
        back = normalized_log_rescale(y.to(DEV), p, clamp)
        r = normalized_log_rescale_oracle(y.numpy(), a, b, clamp)
        assert np.isnan(r).sum() == 1
        assert_matches(back, r, rtol=3e-5)


# ------------------------------------------------------------------------------------------------ mirmap2envmap

def mirmap_bound(m, out_shape, peak):
    """2e-5 of the peak, plus the ill-conditioning of the reference's own formula near the envmap's back seam: there
    h = dir + view is a cancellation (z = 1 - sin(theta) cos(phi)), so fp32 carries an absolute error of a few ulp of 1
    in h_z (bounded here by 8 * 2^-24: sinf, cosf, the product and the sum).  A direction error dz moves the sample by
    W/pi * dz / |h_xz| texels in x and H/pi * dz / |h| in y, which changes the value by at most that times the
    largest step between neighbouring texels.  At 1000 x 2000 the seam's columns come within 2e-3 of h = 0."""
    H, W = m.shape[-2:]
    OH, OW = out_shape
    th, ph = np.meshgrid((np.arange(OH) + 0.5) * (np.pi / OH), -(np.arange(OW) + 0.5) * (2 * np.pi / OW), indexing="ij")
    x, y, z = -np.sin(th) * np.sin(ph), np.cos(th), 1 - np.sin(th) * np.cos(ph)
    dz = 8 * 2.0 ** -24
    step = max(np.abs(np.diff(m, axis=-1)).max(initial=0), np.abs(np.diff(m, axis=-2)).max(initial=0))
    return 2e-5 * peak + step * (W / np.pi * dz / np.sqrt(x * x + z * z) + H / np.pi * dz / np.sqrt(x * x + y * y + z * z))


@pytest.mark.parametrize("C", [1, 2, 4])
@pytest.mark.parametrize("mir_shape", [(17, 33), (32, 32), (33, 17)])
@pytest.mark.parametrize("out_shape", [(5, 7), (33, 65), (1000, 2000)])
def test_mirmap2envmap_shapes(C, mir_shape, out_shape):
    g = torch.Generator().manual_seed(C * 7 + mir_shape[0])
    mir = torch.exp(torch.randn(2, C, *mir_shape, generator=g))
    basis = torch.rand(C, *mir_shape, generator=g) + 0.5
    for bs in (None, basis):
        env = mirmap2envmap(mir.to(DEV), out_shape, basis=None if bs is None else bs.to(DEV))
        assert env.shape == (2, C, *out_shape)
        o = mirmap2envmap_oracle(mir.numpy(), out_shape, basis=None if bs is None else bs.numpy())
        m = mir.double().numpy() if bs is None else mir.double().numpy() / bs.double().numpy()
        tol = mirmap_bound(m, out_shape, np.abs(o).max())
        assert (np.abs(env.cpu().double().numpy() - o) <= tol).all()
    r = r0toenvmap(mir.to(DEV), basis.to(DEV))  # default size (H, 2W), channels last
    o = mirmap2envmap_oracle(mir.numpy(), (mir_shape[0], 2 * mir_shape[1]), basis=basis.numpy()).transpose(0, 2, 3, 1)
    assert r.shape == o.shape
    tol = mirmap_bound(mir.double().numpy() / basis.double().numpy(), o.shape[1:3], np.abs(o).max())[None, ..., None]
    assert (np.abs(r.cpu().double().numpy() - o) <= tol).all()


# ------------------------------------------------------------------------------------------------ refmap lookups

def edge_normals(Hr, Wr, n_random, seed):
    """Random unit normals plus the edges: the poles (+-Y), the limb n_z = 0 on both sides (the phi = 0 / pi seam),
    -0.0 components, and directions at exact cell borders and texel centres of an Hr x Wr refmap."""
    g = torch.Generator().manual_seed(seed)
    n = torch.nn.functional.normalize(torch.randn(n_random, 3, generator=g), dim=-1)
    special = [[0, 1, 0], [0, -1, 0], [-0.0, 1, 0], [0, -1, -0.0], [1, 0, 0], [-1, 0, 0], [0.8, 0.6, 0], [-0.8, -0.6, 0],
               [0.8, 0.6, -0.0], [-0.8, 0.6, -0.0], [-0.0, 0.6, 0.8], [0.0, -0.6, 0.8], [-0.0, -0.0, 1], [0, 0, -1]]
    edges = []
    for i in range(Hr + 1):
        for j in range(2 * Wr + 1):
            th, ph = i * np.pi / Hr, j * np.pi / (2 * Wr)  # j even: cell borders; j odd: texel centres
            edges.append([-np.sin(th) * np.cos(ph), np.cos(th), np.sin(th) * np.sin(ph)])
    return torch.cat([n, torch.tensor(special + edges, dtype=torch.float32)])


@pytest.mark.parametrize("C", [1, 2, 4])
@pytest.mark.parametrize("Hr,Wr", [(24, 40), (7, 13), (40, 24)])
def test_refmap_lookup_shapes_and_edges(C, Hr, Wr):
    """The compacted entry with many empty images in `offsets` (the first two, runs of three, the last but one), then
    the dense entry on one image's normals under a mask, in both layouts."""
    g = torch.Generator().manual_seed(C * 31 + Hr)
    counts = [0, 0, 300, 0, 0, 0, 1, 0, 0, 500, 0, 7]
    B = len(counts)
    maps = torch.exp(torch.randn(B, C, Hr, Wr, generator=g))
    parts = [edge_normals(Hr, Wr, c, seed=b) if c else torch.zeros(0, 3) for b, c in enumerate(counts)]
    nrm = torch.cat(parts)
    offsets = torch.zeros(B + 1, dtype=torch.int64)
    offsets[1:] = torch.tensor([len(q) for q in parts]).cumsum(0)
    out = refmap_lookup(maps.to(DEV), nrm.to(DEV), offsets)
    assert out.shape == (len(nrm), C)
    for b in range(B):
        lo, hi = int(offsets[b]), int(offsets[b + 1])
        if hi > lo:
            o = refmap_lookup_oracle(maps[b].numpy(), nrm[lo:hi].numpy())
            assert_matches(out[lo:hi], o, atol=3e-5 * np.abs(o).max())
    b = 9
    lo, hi = int(offsets[b]), int(offsets[b + 1])
    dn = nrm[lo:hi].reshape(1, 1, hi - lo, 3).to(DEV)
    mk = (torch.arange(hi - lo) % 3 != 1).reshape(1, 1, -1).to(DEV)
    img = refmap_lookup_images(maps[b:b + 1].to(DEV), dn, mk, channel_first=False)[0, 0]
    o = refmap_lookup_oracle(maps[b].numpy(), nrm[lo:hi].numpy())
    o[~mk[0, 0].cpu().numpy()] = 0.0
    assert_matches(img, o, atol=3e-5 * np.abs(o).max())
    assert torch.equal(img[mk[0, 0]], out[lo:hi][mk[0, 0]]) and not img[~mk[0, 0]].any()
    chw = refmap_lookup_images(maps[b:b + 1].to(DEV), dn.permute(0, 3, 1, 2), mk, channel_first=True)
    assert torch.equal(chw[0, :, 0].T, img)


def test_refmap_lookup_dense_beyond_the_grid_y_limit():
    """B = 70 000 images of 4 x 4: the grid covers 65 535 images and loops for the rest.  Images 0, 65 534 .. 65 536 and
    the last against the oracle, all of them bit for bit against the compacted entry."""
    B, H, W, C, Hr, Wr = 70000, 4, 4, 2, 7, 13
    g = torch.Generator().manual_seed(70)
    maps = torch.exp(torch.randn(B, C, Hr, Wr, generator=g)).to(DEV)
    nrm = torch.nn.functional.normalize(torch.randn(B, H, W, 3, generator=g), dim=-1).to(DEV)
    mask = (torch.rand(B, H, W, generator=g) > 0.3).to(DEV)
    mask[65535] = True
    mask[65536] = False
    out = refmap_lookup_images(maps, nrm, mask, channel_first=False)
    offsets = torch.zeros(B + 1, dtype=torch.int64, device=DEV)
    offsets[1:] = mask.sum((1, 2)).cumsum(0)
    comp = refmap_lookup(maps, nrm[mask], offsets)
    assert torch.equal(out[mask], comp) and not out[~mask].any()
    for b in (0, 65534, 65535, 65536, B - 1):
        mb = mask[b].cpu()
        o = refmap_lookup_oracle(maps[b].cpu().numpy(), nrm[b].cpu()[mb].numpy())
        assert_matches(out[b].cpu()[mb], o, atol=3e-5 * np.abs(o).max(initial=1.0))
        assert not out[b].cpu()[~mb].any()


# ------------------------------------------------------------------------------------------------ img2refmap, C != 3

SYNTH = ["A_half_cell_res32", "B_small_window_res64", "C_overlap_res256", "D_min_points_res32", "E_nan_ties_res16",
         "G_nan_angles_res16", "F_wide_window_res24"]


def colours_with(colors, C, seed):
    """The case's colours with one channel, two, or a fourth channel that is NaN for about 3% of the pixels (their sum
    is NaN: they count as members but are never selected nor averaged)."""
    if C < 3:
        return np.ascontiguousarray(colors[:, :C])
    rng = np.random.default_rng(seed)
    a = rng.random((len(colors), 1)).astype(np.float32)
    a[rng.random(len(colors)) < 0.03] = np.nan
    return np.ascontiguousarray(np.concatenate([colors, a], 1))


def same(ours, ref):
    for x, y in zip(ours, ref):
        x = x.cpu().numpy() if isinstance(x, torch.Tensor) else x
        assert x.shape == y.shape and np.array_equal(x, y, equal_nan=x.dtype.kind == "f")


@pytest.mark.parametrize("name", SYNTH)
@pytest.mark.parametrize("C", [1, 2, 4])
def test_img2refmap_channel_counts(golden_synth, name, C):
    """Both entries against img2refmap_oracle bit for bit, median and mean.  The batch entry takes the case as image 1
    of three (image 0 another case, image 2 empty); the dense entry reads the same pixels through strided views."""
    c, other = golden_synth[name], golden_synth["A_half_cell_res32"]
    res, thr, mp = int(c["res"]), float(c["thr"]), int(c["min_points"])
    col, tp = colours_with(c["colors"], C, seed=C), c["thetaphi_torch_cpu"]
    col0, tp0 = colours_with(other["colors"], C, seed=C + 10), other["thetaphi_torch_cpu"]
    colors, thetaphi = np.concatenate([col0, col]), np.concatenate([tp0, tp])
    offsets = np.array([0, len(col0), len(colors), len(colors)])
    for reduce in ("median", "mean"):
        ours = img2refmap_batch(torch.from_numpy(colors).to(DEV), None, torch.from_numpy(offsets), res, thr, mp,
                                thetaphi=torch.from_numpy(thetaphi).to(DEV), reduce=reduce)
        ref = img2refmap_batch_oracle(colors, None, offsets, res, thr, mp, thetaphi=thetaphi, reduce=reduce)
        same(ours, ref)
    # dense: the case's pixels at random positions of a 96 x 112 image, normals from the case (NaN where its angles
    # are NaN); the oracle takes the device's angles of those normals
    n = c["normals"].copy()
    n[np.isnan(tp).any(1)] = np.nan
    H, W = 96, 112
    rng = np.random.default_rng(C)
    pos = np.sort(rng.choice(H * W, len(col), replace=False))
    dc = np.full((H * W, C + 1), np.nan, np.float32)  # one spare channel: the colours are a strided channel slice
    dn = np.zeros((H * W, 3), np.float32)
    dc[pos, :C], dn[pos] = col, n
    mask = np.zeros(H * W, bool)
    mask[pos] = True
    dev_n = torch.from_numpy(n).to(DEV)
    tp_dev = normals_to_thetaphi(dev_n).cpu().numpy()
    dcol = torch.from_numpy(dc.reshape(1, H, W, C + 1)).to(DEV)[..., :C]
    dnrm = torch.from_numpy(dn.reshape(1, H, W, 3)).to(DEV)
    dmask = torch.from_numpy(mask.reshape(1, H, W)).to(DEV)
    for channel_first in (False, True):
        cc = dcol.permute(0, 3, 1, 2) if channel_first else dcol
        nn_ = dnrm.permute(0, 3, 1, 2) if channel_first else dnrm
        for reduce in ("median", "mean"):
            ours = img2refmap_images(cc, nn_, dmask, res, thr, mp, channel_first=channel_first, reduce=reduce)
            o = img2refmap_oracle(col, None, res, thr, mp, thetaphi=tp_dev, reduce=reduce)
            sel = o[3].copy()
            sel[sel >= 0] = pos[sel[sel >= 0]]  # compacted index -> dense y * W + x
            if reduce == "mean":
                sel[:] = -1
            same([t[0] for t in ours], (*o[:3], sel))


# ------------------------------------------------------------------------------------------------ the 2^26 boundary

def spy_on(monkeypatch, entry):
    import drmnet_b200.img2refmap as M
    calls, real = [], M._lib.lib()

    class Spy:
        def __getattr__(self, name):
            return getattr(real, name)

    def call(*args):
        calls.append(args)
        return getattr(real, entry)(*args)

    spy = Spy()
    setattr(spy, entry, call)
    monkeypatch.setattr(M._lib, "lib", lambda: spy)
    return calls


def sphere_512(seed):
    """A 512^2 sphere normal image (about 206k pixels in its mask) with smooth HDR-like colours plus noise."""
    n, m = sphere_normals(256)
    rng = np.random.default_rng(seed)
    col = (np.exp(1.5 * n[..., :1] + 0.7 * n[..., 1:2]) * np.array([1.0, 0.9, 0.8])
           * (1 + 0.01 * rng.standard_normal((512, 512, 3)))).astype(np.float32)
    return col, n.astype(np.float32), m


def test_img2refmap_dense_call_of_exactly_2_26_pixels(monkeypatch):
    """256 images of 512^2 = 2^26 pixels in one call (pixel index 2^26 - 1 is the last that fits below the cell tag);
    empty masks except the last two images."""
    import drmnet_b200.img2refmap as M
    B, res, thr = 256, 128, float(np.pi / 256)
    assert B * 512 * 512 == M.MAX_PIXELS_PER_CALL == 1 << 26
    c0, n0, m0 = sphere_512(1)
    c1, n1, m1 = sphere_512(2)
    colors = torch.from_numpy(c0).to(DEV)[None].repeat(B, 1, 1, 1)
    normals = torch.from_numpy(n0).to(DEV)[None].repeat(B, 1, 1, 1)
    colors[-1], normals[-1] = torch.from_numpy(c1).to(DEV), torch.from_numpy(n1).to(DEV)
    mask = torch.zeros(B, 512, 512, dtype=torch.bool, device=DEV)
    mask[-2], mask[-1] = torch.from_numpy(m0).to(DEV), torch.from_numpy(m1).to(DEV)
    calls = spy_on(monkeypatch, "drm_img2refmap_dense")
    out = img2refmap_images(colors, normals, mask, res, thr, channel_first=False, check_status=True)
    assert len(calls) == 1 and img2refmap_images.last_status[0] == 0
    alone = img2refmap_images(colors[-1:], normals[-1:], mask[-1:], res, thr, channel_first=False)
    same([t[-1] for t in out], [t[0].cpu().numpy() for t in alone])
    assert not out[1][:-2].any() and out[1][-2].any()
    tp = normals_to_thetaphi(normals[-1][mask[-1]]).cpu().numpy()
    o = img2refmap_oracle(c1[m1], None, res, thr, thetaphi=tp)
    sel = o[3].copy()
    sel[sel >= 0] = np.flatnonzero(m1)[sel[sel >= 0]]
    same([t[-1] for t in out], (*o[:3], sel))


def test_img2refmap_batch_call_of_exactly_2_26_pixels(monkeypatch):
    """total_n = 2^26 in one call: image 0 is filler whose angles fall in no cell, image 1 a sphere at the end of the
    pixel range."""
    res, thr = 128, float(np.pi / 256)
    c1, n1, m1 = sphere_512(3)
    col1 = torch.from_numpy(c1[m1]).to(DEV)
    tp1 = normals_to_thetaphi(torch.from_numpy(n1[m1]).to(DEV))
    n_img1 = col1.shape[0]
    total = 1 << 26
    colors = torch.zeros(total, 3, device=DEV)
    thetaphi = torch.empty(total, 2, device=DEV)
    thetaphi[:, 0], thetaphi[:, 1] = np.pi / 2, -np.pi / 2  # phi < 0: behind the refmap, in no cell
    colors[-n_img1:], thetaphi[-n_img1:] = col1, tp1
    offsets = torch.tensor([0, total - n_img1, total], dtype=torch.int64)
    calls = spy_on(monkeypatch, "drm_img2refmap")
    out = img2refmap_batch(colors, None, offsets, res, thr, thetaphi=thetaphi, check_status=True)
    assert len(calls) == 1 and img2refmap_batch.last_status[0] == 0
    assert not out[1][0].any() and int(out[2][0].sum()) == 0
    alone = img2refmap_batch(col1, None, torch.tensor([0, n_img1]), res, thr, thetaphi=tp1)
    same([t[1] for t in out], [t[0].cpu().numpy() for t in alone])
    o = img2refmap_oracle(c1[m1], None, res, thr, thetaphi=tp1.cpu().numpy())
    same([t[1] for t in out], o)
