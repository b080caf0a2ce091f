"""Drop-in for the reference's utils/img2refmap.py on B200: same function name, arguments, returns and errors.

``refmap_mask_make`` (reference utils/img2refmap.py:6-37) bins masked object-image pixels by surface normal into a
res x res refmap and copies, per cell, the pixel with the lower-median channel sum.  The work is done by
``drm_img2refmap`` in libdrmrender.so (hand-written sm_100a kernels, include/drmrender.h); tensors must live on a CUDA
device -- there is no CPU path.  ``img2refmap_batch`` scatters a batch of compacted pixel lists, ``img2refmap_images``
a batch of dense images under a mask (``drm_img2refmap_dense``, read in place).
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} is on {t.device}: drmnet_b200 has no CPU path (CUDA tensors only)")


MAX_PIXELS_PER_CALL = 1 << 26  # include/drmrender.h: a pair keeps its cell tag above a 26-bit pixel index


def split_batch(offsets_host, max_pixels: int = MAX_PIXELS_PER_CALL):
    """Image ranges [(b0, b1), ...] whose pixel totals fit one library call (host logic, no device work)."""
    offs = [int(o) for o in offsets_host]
    groups, b0 = [], 0
    for b in range(len(offs) - 1):
        if offs[b + 1] - offs[b] > max_pixels:
            raise ValueError(f"image {b} has {offs[b + 1] - offs[b]} pixels; one image can hold at most {max_pixels}")
        if offs[b + 1] - offs[b0] > max_pixels:
            groups.append((b0, b))
            b0 = b
    groups.append((b0, len(offs) - 1))
    return groups


def img2refmap_batch(colors: torch.Tensor, normals: torch.Tensor, offsets: torch.Tensor, res: int,
                     angle_threshold: float, min_points: int = 0, *, thetaphi: torch.Tensor | None = None,
                     reduce: str = "median", check_status: bool = False):
    """Segmented scatter of B images in one launch sequence.

    colors [total_n, C] fp32, normals [total_n, 3] fp32 (or ``thetaphi`` [total_n, 2]), offsets [B+1] int64 (image b
    owns rows offsets[b]:offsets[b+1]).  Returns (refmap [B,res,res,C] fp32, refmask [B,res,res] bool,
    counts [B,res,res] int32, sel_index [B,res,res] int32 image-local, -1 where empty).
    ``check_status`` reads the library's status word back (one stream synchronisation) and raises if the pair buffer
    overflowed; ``img2refmap_batch.last_status`` then holds (flags, cells on the warp-per-cell path).
    """
    if isinstance(colors, torch.Tensor) and colors.dim() == 2 and colors.shape[0] > MAX_PIXELS_PER_CALL:
        geom_all = thetaphi if thetaphi is not None else normals
        offs_h = offsets.cpu().tolist()
        parts = []
        for b0, b1 in split_batch(offs_h, MAX_PIXELS_PER_CALL):
            lo, hi = offs_h[b0], offs_h[b1]
            sub = torch.as_tensor(offs_h[b0:b1 + 1], dtype=torch.int64) - lo
            kw = dict(thetaphi=geom_all[lo:hi]) if thetaphi is not None else {}
            parts.append(img2refmap_batch(colors[lo:hi], None if thetaphi is not None else geom_all[lo:hi], sub, res,
                                          angle_threshold, min_points, reduce=reduce, check_status=check_status, **kw))
        return tuple(torch.cat([p[i] for p in parts]) for i in range(4))
    _require_cuda(colors, "colors")
    geom = thetaphi if thetaphi is not None else normals
    _require_cuda(geom, "normals")
    if angle_threshold is None:
        # the reference fails at `angles > angle_threshold` (utils/img2refmap.py:27)
        raise TypeError("'>' not supported between instances of 'Tensor' and 'NoneType'")
    if colors.dtype != torch.float32 or geom.dtype != torch.float32:
        raise TypeError("colors and normals must be float32")
    if colors.dim() != 2 or geom.dim() != 2 or geom.shape[0] != colors.shape[0]:
        raise ValueError(f"colors {tuple(colors.shape)} / normals {tuple(geom.shape)}: expected [n,C] and [n,3]")
    if geom.shape[1] != (2 if thetaphi is not None else 3):
        raise ValueError("normals must be [n,3] (thetaphi [n,2])")
    mode = {"median": 0, "mean": 1}[reduce]
    device = colors.device
    colors = colors.contiguous()
    geom = geom.contiguous()
    offsets = offsets.to(device=device, dtype=torch.int64).contiguous()
    B = offsets.numel() - 1
    total_n, C = colors.shape
    L = _lib.lib()
    with torch.cuda.device(device):
        refmap = torch.empty((B, res, res, C), dtype=torch.float32, device=device)
        refmask = torch.empty((B, res, res), dtype=torch.bool, device=device)  # the kernels store 0/1 bytes
        counts = torch.empty((B, res, res), dtype=torch.int32, device=device)
        sel = torch.empty((B, res, res), dtype=torch.int32, device=device)
        nbytes = L.drm_img2refmap_workspace_bytes(total_n, B, res, float(angle_threshold))
        ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)
        _lib.check(L.drm_img2refmap(colors.data_ptr(), geom.data_ptr(), int(thetaphi is not None), offsets.data_ptr(),
                                    total_n, B, C, int(res), float(angle_threshold), int(min_points), mode,
                                    refmap.data_ptr(), refmask.data_ptr(), counts.data_ptr(), sel.data_ptr(),
                                    ws.data_ptr(), ws.numel(), _stream_ptr(device)))
        if check_status:
            st = (ctypes.c_int32 * 2)()
            _lib.check(L.drm_img2refmap_status(ws.data_ptr(), total_n, B, int(res), float(angle_threshold),
                                               ctypes.byref(st), _stream_ptr(device)))
            img2refmap_batch.last_status = (int(st[0]), int(st[1]))
            if st[0] & 1:
                raise RuntimeError("img2refmap: the (cell, pixel) pair buffer overflowed; outputs are invalid")
        ws.record_stream(torch.cuda.current_stream(device))
    return refmap, refmask, counts, sel


def img2refmap_images(colors: torch.Tensor, normals: torch.Tensor, mask: torch.Tensor | None, res: int,
                      angle_threshold: float, min_points: int = 0, *, channel_first: bool, reduce: str = "median",
                      check_status: bool = False):
    """``img2refmap_batch`` on dense images under a mask, read in place: no compaction, no copy, no host synchronisation.

    colors [B,C,H,W] and normals [B,3,H,W] (``channel_first``) or [B,H,W,C] and [B,H,W,3], fp32, any strides (views
    such as a channel slice or a permute are read through their strides); mask [B,H,W] bool, or None for every pixel.
    A single image without the batch dimension is accepted, and its outputs then have none either.  Bit for bit::

        img2refmap_batch(colors_hwc[mask], normals_hwc[mask], [0, cumsum(mask.sum((1, 2)))], res, angle_threshold, ...)

    except ``sel_index``, which holds the dense image-local index y*W + x of the selected pixel (-1 where empty or in
    mean mode).  Returns (refmap [B,res,res,C], refmask [B,res,res] bool, counts [B,res,res] int32, sel_index).
    The mask is the caller's: build it with the expression the reference uses (e.g. ``normals.norm(dim=1) > 0.5``).
    Batches of more than MAX_PIXELS_PER_CALL pixels (B*H*W, masked or not) are split by whole images on the host.
    ``check_status`` as in ``img2refmap_batch`` (it synchronises).
    """
    _require_cuda(colors, "colors")
    _require_cuda(normals, "normals")
    if angle_threshold is None:
        raise TypeError("'>' not supported between instances of 'Tensor' and 'NoneType'")
    if colors.dtype != torch.float32 or normals.dtype != torch.float32:
        raise TypeError("colors and normals must be float32")
    single = colors.dim() == 3
    if single:
        colors, normals = colors.unsqueeze(0), normals.unsqueeze(0)
        if mask is not None:
            mask = mask.unsqueeze(0)
    if colors.dim() != 4 or normals.dim() != 4:
        raise ValueError(f"colors {tuple(colors.shape)} / normals {tuple(normals.shape)}: expected "
                         f"{'[B,C,H,W] and [B,3,H,W]' if channel_first else '[B,H,W,C] and [B,H,W,3]'}")
    if channel_first:
        B, C, H, W = colors.shape
        dims = (0, 2, 3, 1)  # the (b, y, x, c) strides of a [B,C,H,W] tensor
    else:
        B, H, W, C = colors.shape
        dims = (0, 1, 2, 3)
    if tuple(normals.shape) != ((B, 3, H, W) if channel_first else (B, H, W, 3)):
        raise ValueError(f"normals {tuple(normals.shape)} do not match colors {tuple(colors.shape)}")
    if normals.device != colors.device:
        raise RuntimeError(f"normals are on {normals.device}, colors on {colors.device}")
    if mask is not None:
        _require_cuda(mask, "mask")
        if mask.dtype != torch.bool:
            raise TypeError("mask must be bool")
        if tuple(mask.shape) != (B, H, W) or mask.device != colors.device:
            raise ValueError(f"mask {tuple(mask.shape)} on {mask.device}: expected [{B},{H},{W}] on {colors.device}")
    mode = {"median": 0, "mean": 1}[reduce]
    if B * H * W > MAX_PIXELS_PER_CALL:
        if H * W > MAX_PIXELS_PER_CALL:
            raise ValueError(f"one image has {H * W} pixels; one image can hold at most {MAX_PIXELS_PER_CALL}")
        step = MAX_PIXELS_PER_CALL // (H * W)
        parts = [img2refmap_images(colors[b:b + step], normals[b:b + step], None if mask is None else mask[b:b + step],
                                   res, angle_threshold, min_points, channel_first=channel_first, reduce=reduce,
                                   check_status=check_status) for b in range(0, B, step)]
        return tuple(torch.cat([p[i] for p in parts]) for i in range(4))
    device = colors.device
    L = _lib.lib()
    cs = (ctypes.c_int64 * 4)(*(colors.stride(d) for d in dims))
    ns = (ctypes.c_int64 * 4)(*(normals.stride(d) for d in dims))
    with torch.cuda.device(device):
        mask_u8 = None if mask is None else mask.contiguous().view(torch.uint8)
        refmap = torch.empty((B, res, res, C), dtype=torch.float32, device=device)
        refmask = torch.empty((B, res, res), dtype=torch.bool, device=device)  # the kernels store 0/1 bytes
        counts = torch.empty((B, res, res), dtype=torch.int32, device=device)
        sel = torch.empty((B, res, res), dtype=torch.int32, device=device)
        nbytes = L.drm_img2refmap_dense_workspace_bytes(B, H, W, res, float(angle_threshold))
        ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)
        _lib.check(L.drm_img2refmap_dense(colors.data_ptr(), cs, normals.data_ptr(), ns,
                                          None if mask_u8 is None else mask_u8.data_ptr(), B, H, W, C, int(res),
                                          float(angle_threshold), int(min_points), mode, refmap.data_ptr(),
                                          refmask.data_ptr(), counts.data_ptr(), sel.data_ptr(), ws.data_ptr(),
                                          ws.numel(), _stream_ptr(device)))
        if check_status:
            st = (ctypes.c_int32 * 2)()
            _lib.check(L.drm_img2refmap_status(ws.data_ptr(), B * H * W, B, int(res), float(angle_threshold),
                                               ctypes.byref(st), _stream_ptr(device)))
            img2refmap_images.last_status = (int(st[0]), int(st[1]))
            if st[0] & 1:
                raise RuntimeError("img2refmap: the (cell, pixel) pair buffer overflowed; outputs are invalid")
        ws.record_stream(torch.cuda.current_stream(device))
    out = (refmap, refmask, counts, sel)
    return tuple(o[0] for o in out) if single else out


def refmap_mask_make(colors: torch.Tensor, normals: torch.Tensor, res: int, angle_threshold: float = None,
                     min_points=0, refmap_batch_size=512):
    """Same contract as the reference's refmap_mask_make (utils/img2refmap.py:6-37).

    colors [n,C], normals [n,3] -> (refmap [res,res,C], refmask [res,res] bool).  ``refmap_batch_size`` only chunks
    the reference's dense window test and has no effect on the result; it is accepted and ignored.
    """
    _require_cuda(colors, "colors")
    if colors.shape[0] == 0:
        # torch.nanmedian over an empty dim (utils/img2refmap.py:31)
        raise IndexError("median(): Expected reduction dim 1 to have non-zero size.")
    offsets = torch.tensor([0, colors.shape[0]], dtype=torch.int64, device=colors.device)
    refmap, refmask, _, _ = img2refmap_batch(colors, normals, offsets, res, angle_threshold, min_points)
    return refmap[0], refmask[0]


def normals_to_thetaphi(normals: torch.Tensor) -> torch.Tensor:
    """xyz2thetaphi(normals, normal=[0,1,0], tangent=[-1,0,0]) of utils/transform.py:55-89, on device."""
    _require_cuda(normals, "normals")
    normals = normals.contiguous().float()
    out = torch.empty((normals.shape[0], 2), dtype=torch.float32, device=normals.device)
    with torch.cuda.device(normals.device):
        _lib.check(_lib.lib().drm_normals_to_thetaphi(normals.data_ptr(), normals.shape[0], out.data_ptr(),
                                                      _stream_ptr(normals.device)))
    return out
