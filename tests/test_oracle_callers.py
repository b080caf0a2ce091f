"""Pin the oracles of the 'next' rows (N1 post-processing, N2 mirmap2envmap) on CPU."""
import numpy as np
import torch

from drmnet_b200.synth import sphere_normals
from oracle.callers_oracle import mirmap2envmap_oracle, postprocess_oracle


def test_mirmap2envmap_oracle_matches_reference_output(golden_mirmap):
    """golden: the reference's mirmap2envmap (utils/transform.py:106-144) on its own envmap2mirmap output."""
    mir = golden_mirmap["mirmap_v001"].transpose(2, 0, 1)[None]
    ours = mirmap2envmap_oracle(mir, (32, 64))[0].transpose(1, 2, 0)
    ref = golden_mirmap["envmap_from_mirmap_v001"]
    assert np.abs(ours - ref).max() <= 2e-5 * np.abs(ref).max()


GOLDEN = __import__("pathlib").Path(__file__).resolve().parent / "golden"


def test_postprocess_oracle_matches_reference_code():
    """golden (oracle/gen_golden.py callers_golden): the source lines models/drmnet.py:610-617 executed as they stand,
    then the reference's BaseDataset('log').transform (dataset/basedataset.py:52-53)."""
    g = np.load(GOLDEN / "callers_ref.npz")
    ours, s = postprocess_oracle(g["post_in"])
    assert np.allclose(s, g["post_scale"], rtol=2e-6)
    assert np.allclose(ours, g["post_out"], rtol=2e-6, atol=2e-6)


def test_normalized_log_oracle_matches_reference_code():
    """golden: the reference's BaseDataset('0p1tom1p1_normalizedLogarithmic_lowerbound1e-6').transform with
    dynamic_normalize=True under a mask (dataset/basedataset.py:56-76), imported and run."""
    from oracle.callers_oracle import normalized_log_oracle
    g = np.load(GOLDEN / "callers_ref.npz")
    ours, lmin, lmax = normalized_log_oracle(g["nlog_in"], g["nlog_mask"])
    assert np.allclose(ours, g["nlog_out"], rtol=1e-5, atol=1e-5)
    assert np.allclose(lmin, g["nlog_min"], atol=1e-6) and np.allclose(lmax, g["nlog_max"], atol=1e-6)


def test_postprocess_oracle_matches_torch_formulas():
    """The same expressions evaluated with torch ops (models/drmnet.py:610-620, dataset/basedataset.py:52-53), on finite
    samples and on samples whose LrK holds NaN (scale NaN), +inf (scale 0), -inf (L < 0, excluded) or is all zero (0/0)."""
    g = torch.Generator().manual_seed(0)
    stacks = torch.rand(3, 9, 3, 16, 16, generator=g) * 3
    stacks[0, 1, :, :4] = 0  # L == 0 pixels are excluded from the mean
    stacks[0, 4, 1, 3, 5] = float("nan")
    stacks[0, 5, 0, 7, 7] = float("inf")
    stacks[0, 6, 2, 2, 9] = -float("inf")
    stacks[0, 7] = 0
    stacks[2, 8, 0, 0, 0] = float("nan")  # outside LrK: that element only
    LrK = stacks[0]
    L = 0.212671 * LrK[:, 0] + 0.715160 * LrK[:, 1] + 0.072169 * LrK[:, 2]
    m = L > 0
    Lmean = torch.exp((torch.log(L.clip(1e-5)) * m).sum(dim=(1, 2)) / m.sum(dim=(1, 2)))
    scale = 0.12 / Lmean
    ref = torch.log10(stacks * scale[None, :, None, None, None] + 1e-1) + 1
    with np.errstate(invalid="ignore", divide="ignore"):
        ours, s = postprocess_oracle(stacks.numpy())
    assert np.array_equal(np.isnan(s), [False] * 4 + [True, False, False, True, False]) and s[5] == 0
    assert np.allclose(s, scale.numpy(), rtol=1e-5, equal_nan=True)
    assert np.array_equal(np.isnan(ours), torch.isnan(ref).numpy()) and np.isnan(ours[:, [4, 7]]).all()
    assert np.isnan(ours[:, 8]).sum() == 1 and np.isnan(ours[:, :4]).sum() == 0
    assert np.allclose(ours, ref.numpy(), rtol=1e-5, atol=1e-6, equal_nan=True)


def test_refmap_lookup_oracle_matches_reference_refmap2refimg(golden_mirmap):
    """golden: the reference's refmap2refimg_torch (utils/transform.py:170-198) on a random 32x32 refmap, radius 24."""
    from oracle.callers_oracle import refmap_lookup_oracle
    n, mask = sphere_normals(24)
    assert np.array_equal(mask, golden_mirmap["refimg_mask"])
    ours = refmap_lookup_oracle(golden_mirmap["refimg_refmap"], n[mask])
    ref = golden_mirmap["refimg_image"][:, mask].T
    assert np.abs(ours - ref).max() <= 3e-5 * np.abs(ref).max()


def test_normalized_log_oracle_matches_torch_formulas():
    """dataset/basedataset.py:56-76 evaluated with torch ops, chain lowerbound1e-6 -> normalizedLogarithmic -> 0p1tom1p1.
    Samples 3-6 hold +inf in a masked cell, +inf in an unmasked one (inf * 0), NaN in a masked and in an unmasked cell:
    torch's clip, amax and amin keep the NaN, so each of those samples is NaN throughout; sample 7 has an empty mask."""
    from oracle.callers_oracle import normalized_log_oracle
    g = torch.Generator().manual_seed(2)
    x = torch.exp(torch.randn(8, 3, 16, 16, generator=g) * 2)
    x[0, 0, 0, 0] = 0.0
    mask = (torch.rand(8, 1, 16, 16, generator=g) > 0.3).float()
    mask[3:7, :, 5, 6], mask[3:7, :, 7, 8], mask[7] = 1, 0, 0
    x[3, 2, 5, 6], x[4, 0, 7, 8], x[5, 0, 5, 6], x[6, 2, 7, 8] = float("inf"), float("inf"), float("nan"), float("nan")
    y = torch.clip(x, 1e-6)
    linearmax = (y * mask).amax(dim=(-1, -2, -3), keepdim=True)
    log10max = torch.log10(linearmax)
    log10min = torch.log10((y * mask + (1 - mask) * linearmax).amin(dim=(-1, -2, -3), keepdim=True))
    ref = (torch.log10(y) - log10min) / (log10max - log10min) * 2 - 1
    with np.errstate(invalid="ignore", divide="ignore"):
        ours, lmin, lmax = normalized_log_oracle(x.numpy(), mask.numpy())
    assert torch.isnan(ref[3:8]).all() and not torch.isnan(ref[:3]).any() and np.isnan(lmin[3:7]).all()
    assert np.isneginf(lmin[7]) and np.isneginf(lmax[7])
    assert np.array_equal(np.isnan(ours), torch.isnan(ref).numpy())
    assert np.allclose(ours, ref.numpy(), rtol=1e-5, atol=1e-5, equal_nan=True)
    assert np.allclose(lmin, log10min.reshape(-1).numpy(), atol=1e-6, equal_nan=True)
    assert np.allclose(lmax, log10max.reshape(-1).numpy(), atol=1e-6, equal_nan=True)


def test_obsnet_condition_oracles_match_reference_code():
    """golden: BaseDataset.transform with stored parameters, BaseDataset.rescale (with and without clamp_before_exp), and
    the source lines models/obsnet.py:663-695 (get_cond_for_predict, cond_stage_key 'raw_refmap') executed as they stand
    with the noise they drew recorded -- the plain case and noisy_observe 0.05 + padding 'noise'."""
    from oracle.callers_oracle import (normalized_log_apply_oracle, normalized_log_rescale_oracle,
                                       obsnet_condition_oracle)
    g = np.load(GOLDEN / "callers_ref.npz")
    lmin, lmax = g["nlog_min"], g["nlog_max"]
    assert np.allclose(normalized_log_apply_oracle(g["nlog_fixed_in"], lmin, lmax), g["nlog_fixed_out"], rtol=1e-5, atol=1e-5)
    assert np.allclose(normalized_log_rescale_oracle(g["nlog_rescale_in"], lmin, lmax), g["nlog_rescale_out"], rtol=2e-5)
    assert np.allclose(normalized_log_rescale_oracle(g["nlog_rescale_in"], lmin, lmax, 0.5), g["nlog_rescale_clamped_out"],
                       rtol=2e-5)
    assert g["nlog_rescale_clamped_out"].max() <= 10 ** 0.5 * (1 + 1e-6) < g["nlog_rescale_out"].max()
    cond, a, b = obsnet_condition_oracle(g["nlog_in"], g["nlog_mask"])
    assert np.allclose(cond, g["cond_plain"], rtol=1e-5, atol=1e-5) and np.allclose(a, lmin, atol=1e-6)
    assert np.array_equal(g["cond_plain_mask"], g["nlog_mask"].astype(np.float32))
    cond, _, _ = obsnet_condition_oracle(g["nlog_in"], g["nlog_mask"], noisy_observe=0.05,
                                         observe_noise=g["cond_noisy_noise0"], padding_noise=g["cond_noisy_noise1"])
    assert np.allclose(cond, g["cond_noisy"], rtol=1e-5, atol=1e-5)
    outside = ~np.broadcast_to(g["nlog_mask"], cond.shape)
    assert np.allclose(cond[outside], (0.05 * g["cond_noisy_noise0"] + g["cond_noisy_noise1"])[outside], atol=1e-6)
