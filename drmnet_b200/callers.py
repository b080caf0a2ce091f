"""Batched fast paths for the reference's callers of the renderer (SURVEY 8f N1, N2): one launch sequence per training
step instead of one synchronous render per (sample, BRDF vector).

* ``rendering_refmaps``  <- DRMNet.rendering_refmaps          (models/drmnet.py:667-705)
* ``synthesize_refmaps`` <- the render + normalise + transform part of DRMNet.get_input  (models/drmnet.py:523-569,
                            :610-620; dataset/basedataset.py:52-53), NaN-sentinel protocol included
* ``refmap_postprocess`` <- models/drmnet.py:610-620 alone
* ``mirmap2envmap`` / ``r0toenvmap`` <- utils/transform.py:106-144 / DRMNet.r0toenvmap (models/drmnet.py:931-941)
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from .renderer import B200RefMapRenderer, _env_dtype, _slots, render_batch


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def rendering_refmaps(renderer: B200RefMapRenderer, envmaps, z: torch.Tensor,
                      brdf_param_names: Optional[Sequence[str]] = None, view_from=None,
                      new_scene: bool = False) -> torch.Tensor:
    """envmaps [B,He,We,3] (a tensor, or a list of [He,We,3] tensors), z [L,B,P] -> [L,B,3,res,res]: the L BRDF vectors
    of sample b share envmap b and view b, exactly the grouping of the reference's double loop
    (models/drmnet.py:680-705), in one batched launch.  ``view_from`` is [B,3] or a list of B views.  fp16 envmaps are
    rendered in place and the renderer keeps the last one in fp16 (see ``render_batch``: fp16 ends at 65504).

    Like the loop it replaces, the call leaves its mark on the stateful renderer when ``new_scene`` is false: parameters
    that are not named come from the renderer's persistent BSDF, and afterwards the renderer holds the last envmap, the
    last view and the last BRDF vector (utils/mitsuba3_utils.py:411-430 called with envmap/view only at list_idx 0)."""
    assert len(envmaps) == z.size(1)
    if isinstance(envmaps, (list, tuple)):
        if isinstance(envmaps[0], str):
            # the reference's branch for names (models/drmnet.py:685-689) empties the list it iterates and cannot work;
            # EXR reading is outside the render path
            raise NotImplementedError("envmap names are not supported: pass the [He,We,3] tensors")
        envmaps = torch.stack([torch.as_tensor(e) for e in envmaps])
    if isinstance(view_from, (list, tuple)):
        view_from = torch.stack([torch.as_tensor(v, dtype=torch.float32) for v in view_from])
    L, B = z.shape[0], z.shape[1]
    names = brdf_param_names or renderer.brdf_param_names
    device = envmaps.device
    if view_from is None:
        view = (renderer._new_scene_view if new_scene else renderer._view).to(device)[None].expand(B, 3)
    else:
        view = view_from.to(device)
    zz = z.to(device).transpose(0, 1).reshape(B * L, -1)  # batch-major like the reference's iteration order
    flip = renderer._new_scene_flip if new_scene else renderer._flip
    if not new_scene:
        # unnamed parameters keep the persistent scene's values (they cannot change inside the loop either)
        z6 = renderer._bsdf.to(device).repeat(B * L, 1)
        slots = _slots(names)
        z6[:, slots] = zz[:, :len(slots)].float().clip(0, 1)
        zz, names_arg = z6, None
    else:
        names_arg = names
    env_index = torch.arange(B, device=device).repeat_interleave(L)
    out = render_batch(envmaps, zz, view.repeat_interleave(L, dim=0), env_index=env_index, brdf_param_names=names_arg,
                       flip=torch.full((B * L,), bool(flip), device=device), res=renderer.refmap_res,
                       footprint_S=renderer.footprint_S, alpha_min=renderer.alpha_min or 0.0, channel_first=True)
    if not new_scene:
        renderer._envmap = envmaps[-1].to(renderer.device, _env_dtype(envmaps))
        renderer._bsdf = zz[-1].detach().clone()
        if view_from is not None:
            renderer._view = view[-1].detach().float().cpu()
    elif view_from is not None:
        renderer._new_scene_view = view[-1].detach().float().cpu()
    return out.reshape(B, L, 3, renderer.refmap_res, renderer.refmap_res).transpose(0, 1).contiguous()


def refmap_postprocess(stacks: torch.Tensor, refmap_input_scaler: Optional[float] = 0.12, transform: str = "log"
                       ) -> Tuple[torch.Tensor, torch.Tensor]:
    """stacks [G,N,3,res,res] (stack 0 = LrK) -> (normalised + transformed stacks, normalizing_scale [N]).

    One fused kernel for models/drmnet.py:610-620: scale every stack of a sample so the geometric mean of LrK's
    luminance over L > 0 is ``refmap_input_scaler`` (None: no scaling), then log10(x + 0.1) + 1 (``transform="log"``,
    dataset/basedataset.py:52-53; ``None``: identity)."""
    if not stacks.is_cuda:
        raise RuntimeError("stacks must be CUDA tensors: drmnet_b200 has no CPU path")
    if transform not in ("log", None):
        raise NotImplementedError(f"transform {transform!r}: only 'log' (the shipped DRMNet configs) or None")
    stacks = stacks.contiguous().float()
    G, N, C, H, W = stacks.shape
    assert C == 3 and H == W
    out = torch.empty_like(stacks)
    scale = torch.empty(N, dtype=torch.float32, device=stacks.device)
    with torch.cuda.device(stacks.device):
        _lib.check(_lib.lib().drm_refmap_postprocess(stacks.data_ptr(), G, N, H, float(refmap_input_scaler or 0.0),
                                                     1 if transform == "log" else 0, scale.data_ptr(), out.data_ptr(),
                                                     _stream(stacks.device)))
    return out, scale


def synthesize_refmaps(renderer: B200RefMapRenderer, stacked_z: torch.Tensor, envmap,
                       view_from: torch.Tensor, cached: Optional[List[Optional[torch.Tensor]]] = None,
                       brdf_param_names: Optional[Sequence[str]] = None, refmap_input_scaler: Optional[float] = 0.12,
                       transform: str = "log", env_ids: Optional[torch.Tensor] = None):
    """Training-data synthesis of DRMNet.get_input (models/drmnet.py:523-569, 610-620) as two launches.

    stacked_z [G,B,P] (LrK, Lrk, Lrkm1[, r0]); envmap [B,He,We,3]; view_from [B,3]; ``cached[g]`` is either None or a
    [B,3,res,res] tensor whose entries with NaN at [b,0,0,0] are cache misses (the dataset's sentinel,
    dataset/parametricrefmap.py:174-193).  Only misses are rendered.  Returns (list of G transformed [B,3,res,res]
    tensors, normalizing_scale [B], raw stacks [G,B,3,res,res]).

    ``envmap`` may also be an ``EnvmapBank`` of resident maps, with ``env_ids`` [B]: batch element b uses slot
    ``env_ids[b]``, and no map is shipped or re-read per step.  ``env_ids`` applies to an [E,He,We,3] tensor too."""
    G, B = stacked_z.shape[0], stacked_z.shape[1]
    res = renderer.refmap_res
    device = envmap.device
    if env_ids is not None:
        env_ids = torch.as_tensor(env_ids).to(device=device, dtype=torch.int64).reshape(-1)
        if env_ids.numel() != B:
            raise ValueError(f"env_ids has {env_ids.numel()} entries for a batch of {B}")
    raw = torch.empty((G, B, 3, res, res), dtype=torch.float32, device=device)
    need = torch.ones((G, B), dtype=torch.bool, device=device)
    if cached is not None:
        for gi, c in enumerate(cached):
            if c is not None:
                raw[gi] = c.to(device)
                need[gi] = torch.isnan(raw[gi][:, 0, 0, 0])
    idx = torch.nonzero(need.T)  # (batch_idx, stack_idx): the reference's iteration order (models/drmnet.py:561)
    if idx.numel():
        b_idx, g_idx = idx[:, 0], idx[:, 1]
        out = render_batch(envmap, stacked_z.to(device)[g_idx, b_idx], view_from.to(device)[b_idx],
                           env_index=b_idx if env_ids is None else env_ids[b_idx],
                           brdf_param_names=brdf_param_names or renderer.brdf_param_names, res=res,
                           footprint_S=renderer.footprint_S, alpha_min=renderer.alpha_min or 0.0, channel_first=True)
        raw[g_idx, b_idx] = out
    post, scale = refmap_postprocess(raw, refmap_input_scaler, transform)
    return list(post), scale, raw


def mirmap2envmap(mirmap: torch.Tensor, output_shape: tuple, view=[0, 0, 1], basis: Optional[torch.Tensor] = None,
                  log_scale_interpolation: bool = False) -> torch.Tensor:
    """utils/transform.py:106-144 with its defaults: mirmap [B,C,H,W] -> envmap [B,C,OH,OW].  ``basis`` [C,H,W] divides
    the refmap first (fused form of models/drmnet.py:939)."""
    assert list(view) == [0, 0, 1], "now support [0,0,1] view direction"  # the reference's own restriction (:116)
    if log_scale_interpolation:
        raise NotImplementedError("log_scale_interpolation")
    if not mirmap.is_cuda:
        raise RuntimeError("mirmap must be a CUDA tensor: drmnet_b200 has no CPU path")
    mirmap = mirmap.contiguous().float()
    B, C, H, W = mirmap.shape
    OH, OW = output_shape
    out = torch.empty((B, C, OH, OW), dtype=torch.float32, device=mirmap.device)
    bptr = None
    if basis is not None:
        basis = basis.to(mirmap.device).contiguous().float()
        assert tuple(basis.shape) == (C, H, W)
        bptr = basis.data_ptr()
    with torch.cuda.device(mirmap.device):
        _lib.check(_lib.lib().drm_mirmap2envmap(mirmap.data_ptr(), bptr, B, C, H, W, OH, OW, out.data_ptr(),
                                                _stream(mirmap.device)))
    return out


def r0toenvmap(r0: torch.Tensor, basis_r0: torch.Tensor, envshape: Optional[Tuple[int, int]] = None) -> torch.Tensor:
    """DRMNet.r0toenvmap (models/drmnet.py:931-941): r0 [B,C,H,W] rescaled -> envmap [B,OH,OW,3]."""
    if envshape is None:
        envshape = (r0.shape[-2], r0.shape[-1] * 2)
    return mirmap2envmap(r0, envshape, basis=basis_r0).permute(0, 2, 3, 1)


def refmap_lookup(refmap: torch.Tensor, normals: torch.Tensor, offsets: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Shade pixels by their normals: colors [n,C] = bilinear lookup of refmap [B,C,H,W] (or [C,H,W]) at the (theta, phi)
    of normals [n,3]; image b owns rows offsets[b]:offsets[b+1].  The arithmetic of refmap2refimg_torch
    (utils/transform.py:170-198) for arbitrary object normals -- the stand-in for the reference's mesh path tracer in
    the parametric_img2refmap flow (SURVEY 8f N3)."""
    if not refmap.is_cuda:
        raise RuntimeError("refmap must be a CUDA tensor: drmnet_b200 has no CPU path")
    if refmap.dim() == 3:
        refmap = refmap[None]
    refmap = refmap.contiguous().float()
    normals = normals.to(refmap.device).contiguous().float()
    B, C, H, W = refmap.shape
    n = normals.shape[0]
    if offsets is None:
        assert B == 1
        offsets = torch.tensor([0, n], dtype=torch.int64, device=refmap.device)
    offsets = offsets.to(device=refmap.device, dtype=torch.int64).contiguous()
    colors = torch.empty((n, C), dtype=torch.float32, device=refmap.device)
    with torch.cuda.device(refmap.device):
        _lib.check(_lib.lib().drm_refmap_lookup(refmap.data_ptr(), normals.data_ptr(), offsets.data_ptr(), n, B, C, H, W,
                                                colors.data_ptr(), _stream(refmap.device)))
    return colors


def normalized_log_transform(x: torch.Tensor, mask: torch.Tensor, lowerbound: float = 1e-6):
    """ObsNet's conditioning transform `0p1tom1p1_normalizedLogarithmic_lowerbound1e-6` with dynamic_normalize=True
    (dataset/basedataset.py:56-76; models/obsnet.py:224,370): x [B,C,H,W], mask [B,1,H,W] or [B,H,W].
    Returns (out [B,C,H,W] in [-1,1] over the mask, (log10min [B], log10max [B]))."""
    if not x.is_cuda:
        raise RuntimeError("x must be a CUDA tensor: drmnet_b200 has no CPU path")
    x = x.contiguous().float()
    B, C, H, W = x.shape
    mask = mask.to(x.device).float().reshape(B, H, W).contiguous()
    out = torch.empty_like(x)
    lmin = torch.empty(B, dtype=torch.float32, device=x.device)
    lmax = torch.empty(B, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().drm_normalized_log(x.data_ptr(), mask.data_ptr(), B, C, H, W, float(lowerbound),
                                                 out.data_ptr(), lmin.data_ptr(), lmax.data_ptr(), _stream(x.device)))
    return out, (lmin, lmax)


def _nlog_apply(x: torch.Tensor, params, lowerbound: float, inverse: int, clamp_before_exp: float) -> torch.Tensor:
    if not x.is_cuda:
        raise RuntimeError("x must be a CUDA tensor: drmnet_b200 has no CPU path")
    x = x.contiguous().float()
    B, C, H, W = x.shape
    lmin, lmax = (p.to(x.device).float().reshape(-1).contiguous() for p in params)
    if lmin.numel() != B or lmax.numel() != B:
        # the reference asserts the parameters broadcast against x (dataset/basedataset.py:69)
        raise AssertionError(f"{B} samples but {lmin.numel()} / {lmax.numel()} normalisation parameters")
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().drm_normalized_log_apply(x.data_ptr(), lmin.data_ptr(), lmax.data_ptr(), B, C, H, W,
                                                       float(lowerbound), inverse, float(clamp_before_exp or 0.0),
                                                       out.data_ptr(), _stream(x.device)))
    return out


def normalized_log_apply(x: torch.Tensor, params, lowerbound: float = 1e-6) -> torch.Tensor:
    """`ds.transform(x, dynamic_normalize=False)` for `0p1tom1p1_normalizedLogarithmic_lowerbound<lb>` with the parameters
    (log10min [B], log10max [B]) of an earlier dynamic call -- LrK at models/obsnet.py:371 (dataset/basedataset.py:68-72)."""
    return _nlog_apply(x, params, lowerbound, 0, 0.0)


def normalized_log_rescale(y: torch.Tensor, params, clamp_before_exp: float = 0.0) -> torch.Tensor:
    """`ds.rescale(y)` for the same chain (dataset/basedataset.py:83-110): back to linear radiance."""
    return _nlog_apply(y, params, 0.0, 1, clamp_before_exp)


def obsnet_condition(raw_refmap: torch.Tensor, raw_refmask: torch.Tensor, lowerbound: float = 1e-6,
                     noisy_observe: float = 0.0, observe_noise: Optional[torch.Tensor] = None,
                     padding_mode: str = "zeros", padding_noise: Optional[torch.Tensor] = None):
    """ObsNet's conditioning from an observed refmap, one fused kernel (models/obsnet.py:672-691 with
    cond_stage_key "raw_refmap"; the training path :368-370 is noisy_observe=0, padding "zeros").

    raw_refmap [B,C,H,W], raw_refmask [B,H,W] bool/float.  Returns (cond [B,C,H,W], mask [B,1,H,W] float,
    (log10min [B], log10max [B])).  The reference draws its noise with torch.randn_like; pass the tensors
    (``observe_noise`` when noisy_observe > 0, ``padding_noise`` when padding_mode == "noise") or leave them None to
    have them drawn here with torch.randn_like in the reference's order."""
    if padding_mode not in ("zeros", "noise"):
        raise NotImplementedError()  # models/obsnet.py:694-695
    if not raw_refmap.is_cuda:
        raise RuntimeError("raw_refmap must be a CUDA tensor: drmnet_b200 has no CPU path")
    x = raw_refmap.contiguous().float()
    B, C, H, W = x.shape
    mask = raw_refmask.to(x.device).float().reshape(B, H, W).contiguous()
    n1 = n2 = None
    if noisy_observe > 0:
        n1 = torch.randn_like(x) if observe_noise is None else observe_noise.to(x.device).float().contiguous()
    if padding_mode == "noise":
        n2 = torch.randn_like(x) if padding_noise is None else padding_noise.to(x.device).float().contiguous()
    cond = torch.empty_like(x)
    lmin = torch.empty(B, dtype=torch.float32, device=x.device)
    lmax = torch.empty(B, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().drm_obsnet_condition(x.data_ptr(), mask.data_ptr(), B, C, H, W, float(lowerbound),
                                                   float(noisy_observe), n1.data_ptr() if n1 is not None else None,
                                                   n2.data_ptr() if n2 is not None else None, cond.data_ptr(),
                                                   lmin.data_ptr(), lmax.data_ptr(), _stream(x.device)))
    return cond, mask[:, None], (lmin, lmax)
