"""Drop-in for the reference's MitsubaRefMapRenderer (utils/mitsuba3_utils.py:317-430) on B200.

Same constructor keywords, public attributes and ``rendering()`` signature, including the statefulness of the
reference (``None`` for envmap / view_from / flip means "keep the last one", BRDF parameters that are not named keep
their last value in the persistent scene, ``new_scene=True`` renders with a fresh scene).  The image is the
deterministic limit of the reference's Monte-Carlo scene (see DESIGN.md: parity against Mitsuba is unpinned) computed
by ``drm_render_refmaps`` in libdrmrender.so.  Point a config at it with

    renderer_config:
      target: drmnet_b200.renderer.B200RefMapRenderer      # was utils.mitsuba3_utils.MitsubaRefMapRenderer
      params: {refmap_res: 128, spp: 256, denoise: simple, brdf_param_names: [...]}

``render_batch`` is the additive batched entry (one launch for N renders) used by the patched callers of
models/drmnet.py:561-569 and :680-691.
"""
from __future__ import annotations

import ctypes
import math
from typing import List, Optional, Sequence

import torch

from . import _lib

_SLOT = {"metallic.value": 0, "base_color.value.R": 1, "base_color.value.G": 2, "base_color.value.B": 3,
         "roughness.value": 4, "specular": 5}
_SCENE_DEFAULTS = (0.0, 0.0, 0.0, 0.0, 0.0, 1.0)  # utils/mitsuba3_utils.py:348-361


def _slots(names: Sequence[str]) -> List[int]:
    out = []
    for n in names:
        if n not in _SLOT:
            raise NotImplementedError(f"BRDF parameter {n!r}: only {sorted(_SLOT)} are implemented "
                                      "(the parameters DRMNet's configs drive)")
        out.append(_SLOT[n])
    return out


def default_alpha_min(He: int) -> float:
    """Lower clamp of the GGX alpha the library applies when none is given: max(1e-3, 1.25 * pi / He) (DESIGN.md 3)."""
    return max(1e-3, 1.25 * math.pi / He)


def auto_footprint(roughness: float, res: int = 128, alpha_min: float = 1e-3) -> int:
    """Gauss-Legendre points per axis (1, 2, 4, 8 or 16) that resolve the cell average of a GGX lobe of this roughness
    to ~2e-4: the ratio of cell width to lobe half-width decides (measured with the fp64 oracle, DESIGN.md).
    ``alpha_min`` is the clamp the render will apply (``default_alpha_min(He)`` unless the caller overrides it)."""
    alpha = max(float(roughness) ** 2, alpha_min)
    ratio = (math.pi / res) / alpha
    if ratio < 0.1:
        return 1
    if ratio < 0.6:
        return 2
    if ratio < 2.0:
        return 4
    if ratio < 4.0:
        return 8
    return 16


def _env_dtype(envmap: torch.Tensor) -> torch.dtype:
    """Storage type of an envmap on the device: fp16 stays fp16 (the render reads it natively), the rest becomes fp32."""
    return torch.float16 if envmap.dtype == torch.float16 else torch.float32


class EnvmapBank:
    """Envmaps resident on the device with their diffuse pyramids built once (``drm_env_pyramid_build``).

    ``envmaps`` [B,He,We,3] CUDA: fp16 stays fp16 and every other dtype becomes fp32, as in ``render_batch``.  A map
    that is already contiguous in that dtype is used in place, not copied.  Pass the bank to ``render_batch`` (or
    ``synthesize_refmaps``) instead of the maps: ``env_index`` then holds bank slots, and the render reads the pyramids
    instead of building those of the maps it uses on every call.  Its refmaps are bit for bit those of
    ``render_batch`` on the plain maps, and its workspace does not grow with B.

    The diffuse pyramid depends on the texels only, so a bank is built once per map set.  ``update(ids, maps)`` copies
    new maps into slots, ``update(ids)`` re-reads slots changed in place, and both rebuild only those slots.  The bank
    records the version counter of its maps: a render after an in-place change that no ``update`` followed raises
    instead of reading a stale pyramid.  Builds run on the current stream; renders on another stream must wait for
    them."""

    def __init__(self, envmaps: torch.Tensor):
        if not (isinstance(envmaps, torch.Tensor) and envmaps.is_cuda):
            raise RuntimeError("envmaps must be a CUDA tensor: drmnet_b200 has no CPU path")
        if envmaps.dim() != 4 or envmaps.shape[-1] != 3:
            raise ValueError(f"envmaps {tuple(envmaps.shape)}: expected [B,He,We,3]")
        self.maps = envmaps.to(_env_dtype(envmaps)).contiguous()
        self.B, self.He, self.We = (int(s) for s in self.maps.shape[:3])
        self.half = self.maps.dtype == torch.float16
        self.device = self.maps.device
        nbytes = _lib.lib().drm_env_pyramid_bytes(self.B, self.He, self.We)
        if nbytes == 0:
            raise ValueError(f"EnvmapBank: unsupported sizes B={self.B} He={self.He} We={self.We}")
        self.pyramids = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
        self._build(None)

    def _build(self, ids: Optional[torch.Tensor]) -> None:
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().drm_env_pyramid_build(
                self.maps.data_ptr(), int(self.half), self.B, self.He, self.We,
                ids.data_ptr() if ids is not None else None, ids.numel() if ids is not None else 0,
                self.pyramids.data_ptr(), self.pyramids.numel(), torch.cuda.current_stream(self.device).cuda_stream))
        self._version = self.maps._version

    def update(self, ids, maps: Optional[torch.Tensor] = None) -> None:
        """Rebuild the pyramids of slots ``ids`` (a list or an int tensor).  With ``maps``
        [len(ids),He,We,3] the maps are first copied into those slots (converted to the bank's dtype); without, the
        slots are re-read as they are, after the caller changed them in place.  ``update`` declares that no other slot
        changed: the bank's version counter is taken as current afterwards."""
        ids_host = torch.as_tensor(ids, dtype=torch.int64).reshape(-1).cpu()
        if ids_host.numel() and (int(ids_host.min()) < 0 or int(ids_host.max()) >= self.B):
            raise IndexError(f"EnvmapBank.update: slots must be in [0, {self.B})")
        if ids_host.unique().numel() != ids_host.numel():
            raise ValueError("EnvmapBank.update: repeated slot")
        if ids_host.numel() == 0:  # an empty device tensor has a null pointer, which the build reads as "every slot"
            self._version = self.maps._version
            return
        dev_ids = ids_host.to(self.device)
        if maps is not None:
            if tuple(maps.shape) != (ids_host.numel(), self.He, self.We, 3):
                raise ValueError(f"EnvmapBank.update: maps {tuple(maps.shape)}, expected "
                                 f"[{ids_host.numel()},{self.He},{self.We},3]")
            self.maps.index_copy_(0, dev_ids, maps.to(self.device, self.maps.dtype))
        self._build(dev_ids.to(torch.int32))

    @property
    def stale(self) -> bool:
        """True when the maps changed in place since the last build or ``update``."""
        return self.maps._version != self._version

    def check_fresh(self) -> None:
        if self.stale:
            raise RuntimeError("EnvmapBank: the maps changed in place after the pyramids were built; call "
                               "update(ids) with the changed slots before rendering")


def render_batch(envmaps, z: torch.Tensor, view_from: torch.Tensor, *,
                 env_index: Optional[torch.Tensor] = None, flip: Optional[torch.Tensor] = None,
                 brdf_param_names: Optional[Sequence[str]] = None, res: int = 128, footprint_S=1,
                 alpha_min: float = 0.0, channel_first: bool = True, out: Optional[torch.Tensor] = None,
                 options=None, flat: bool = False, check_status: bool = False) -> torch.Tensor:
    """N renders in one launch.  envmaps [B,He,We,3] fp32 or fp16 CUDA; z [N,P]; view_from [N,3]; env_index [N] int
    (default arange, needs N == B); flip [N] bool; footprint_S 1, 2, 4, 8 or 16: an int, one per render, or None (chosen per
    render from its roughness by ``auto_footprint``).  Returns [N,3,res,res] (or [N,res,res,3]).

    ``options``: a ``_lib.RenderOptions`` (accuracy / cost constants, default ``_lib.default_render_options()``).
    ``flat=True`` evaluates the same sum pair by pair (``drm_render_refmaps_flat``, the validation path; any S in 1..16).
    ``check_status=True`` synchronises and raises if a traversal list overflowed or an env_index was out of range.

    An fp16 envmap is read in place (``drm_render_refmaps_half``: no fp32 copy) and gives bit for bit the result of its
    fp32 upcast.  fp16 ends at 65504: brighter texels (a sun) become inf, so convert with ``env.clamp(max=65504).half()``.
    ``flat=True`` and every other dtype render an fp32 copy.

    ``envmaps`` may be an ``EnvmapBank``: ``env_index`` then holds its slots, and the render reads the bank's diffuse
    pyramids (``drm_render_refmaps_prepared``) with the same result.  ``flat=True`` renders the bank's maps as before."""
    bank = None
    if isinstance(envmaps, EnvmapBank):
        envmaps.check_fresh()
        if not flat:
            bank = envmaps
        envmaps = envmaps.maps
    if not (isinstance(envmaps, torch.Tensor) and envmaps.is_cuda):
        raise RuntimeError("envmaps must be a CUDA tensor: drmnet_b200 has no CPU path")
    if envmaps.dim() != 4 or envmaps.shape[-1] != 3:
        raise ValueError(f"envmaps {tuple(envmaps.shape)}: expected [B,He,We,3]")
    device = envmaps.device
    half = envmaps.dtype == torch.float16 and not flat
    envmaps = envmaps.contiguous() if half else envmaps.contiguous().float()
    B, He, We, _ = envmaps.shape
    z = z.to(device=device, dtype=torch.float32)
    if z.dim() != 2:
        raise ValueError("z must be [N,P]")
    N = z.shape[0]
    if brdf_param_names is None:
        if z.shape[1] != 6:
            raise ValueError("z must have 6 columns when brdf_param_names is not given")
        z6 = z.contiguous()
    else:
        slots = _slots(brdf_param_names)
        z6 = torch.tensor(_SCENE_DEFAULTS, device=device).repeat(N, 1)
        z6[:, slots] = z[:, :len(slots)]
    view_from = view_from.to(device=device, dtype=torch.float32).reshape(-1, 3)
    if view_from.shape[0] == 1 and N > 1:
        view_from = view_from.expand(N, 3)
    view_from = view_from.contiguous()
    if view_from.shape[0] != N:
        raise ValueError("view_from must be [N,3]")
    shape = (N, 3, res, res) if channel_first else (N, res, res, 3)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=device)
    elif tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_contiguous():
        raise ValueError("out has the wrong shape/dtype/layout")
    if env_index is None:
        if N != B:
            raise ValueError("env_index is required when N != B")
        env_index = torch.arange(N, dtype=torch.int32, device=device)
    else:
        env_index = env_index.to(device=device, dtype=torch.int32).contiguous()
    if flip is not None:
        flip = flip.to(device=device, dtype=torch.uint8).contiguous()

    # footprint: one S for the whole batch, one per render, or None = chosen per render from its roughness.  The
    # hierarchical path takes all three in ONE launch sequence (the choice is made on the device: no host read of z);
    # the single-level validation path runs one launch per distinct S.
    per_render = None
    if footprint_S is None:
        S_call = 0
    elif isinstance(footprint_S, int):
        S_call = int(footprint_S)
    else:
        per_render = footprint_S if isinstance(footprint_S, torch.Tensor) else torch.tensor([int(s) for s in footprint_S])
        if per_render.numel() != N:
            raise ValueError("footprint_S must be an int or have one entry per render")
        per_render = per_render.to(device=device, dtype=torch.int32).contiguous()
        S_call = 0
    stream = torch.cuda.current_stream(device).cuda_stream
    L = _lib.lib()

    def common_args(S, zz, vv, ee, ff, oo, ws):
        return (envmaps.data_ptr(), B, He, We, ee.data_ptr(), zz.data_ptr(), vv.data_ptr(),
                ff.data_ptr() if ff is not None else None, zz.shape[0], int(res), int(S), float(alpha_min),
                int(channel_first), oo.data_ptr(), ws.data_ptr(), ws.numel(), stream)

    with torch.cuda.device(device):
        if flat:
            if footprint_S is None:
                amin = alpha_min if alpha_min and alpha_min > 0 else default_alpha_min(He)
                S_list = [auto_footprint(r, res, amin) for r in z6[:, 4].clip(0, 1).tolist()]
            elif per_render is not None:
                S_list = per_render.tolist()
            else:
                S_list = [S_call] * N
            for S in sorted(set(S_list)):
                ids = torch.tensor([i for i, s in enumerate(S_list) if s == S], device=device)
                nbytes = L.drm_render_flat_workspace_bytes(ids.numel(), B, He, We, int(res), int(S))
                if nbytes == 0:
                    raise ValueError(f"render_batch: unsupported sizes N={ids.numel()} B={B} He={He} We={We} res={res} S={S}")
                ws = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
                part = out if len(set(S_list)) == 1 else torch.empty((ids.numel(),) + shape[1:], dtype=torch.float32, device=device)
                _lib.check(L.drm_render_refmaps_flat(*common_args(
                    S, z6[ids].contiguous(), view_from[ids].contiguous(), env_index[ids].contiguous(),
                    flip[ids].contiguous() if flip is not None else None, part, ws)))
                if part is not out:
                    out.index_copy_(0, ids, part)
            return out
        ws_bytes = L.drm_render_prepared_workspace_bytes if bank is not None else L.drm_render_workspace_bytes
        nbytes = ws_bytes(N, B, He, We, int(res), 0 if per_render is not None else S_call)
        if nbytes == 0:
            raise ValueError(f"render_batch: unsupported sizes N={N} B={B} He={He} We={We} res={res} S={footprint_S} "
                             "(footprints are 1, 2, 4, 8 or 16)")
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        o = options
        if per_render is not None:
            o = _lib.RenderOptions()
            ctypes.memmove(ctypes.byref(o), ctypes.byref(options if options is not None else _lib.default_render_options()),
                           ctypes.sizeof(o))
            o.footprint_per_render = per_render.data_ptr()
        opts = ctypes.byref(o) if o is not None else None
        if bank is not None:
            _lib.check(L.drm_render_refmaps_prepared(envmaps.data_ptr(), int(half), bank.pyramids.data_ptr(),
                                                     bank.pyramids.numel(),
                                                     *common_args(S_call, z6, view_from, env_index, flip, out, ws)[1:],
                                                     opts))
        else:
            render = L.drm_render_refmaps_half if half else L.drm_render_refmaps_opts
            _lib.check(render(*common_args(S_call, z6, view_from, env_index, flip, out, ws), opts))
        if check_status:
            st = (ctypes.c_int * 40)()
            _lib.check(L.drm_render_status(ws.data_ptr(), st, stream))
            torch.cuda.current_stream(device).synchronize()
            render_batch.last_status = list(st)
            if st[0]:
                raise RuntimeError(f"render_batch: status {st[0]} (1: hand-over pool exhausted, 2: env_index out of range, "
                                   f"4: traversal stack overflow, 8: a footprint was not 1, 2, 4, 8 or 16); "
                                   f"high-water marks {list(st)[1:]}")
    return out


class B200RefMapRenderer:
    """Same interface as MitsubaRefMapRenderer (utils/mitsuba3_utils.py:317-339, 411-430).

    ``rendering`` keeps an fp16 envmap in fp16 (half the memory, the same image as its fp32 upcast; see ``render_batch``
    for the 65504 limit) and converts every other dtype to fp32.  The persistent envmap is kept as an ``EnvmapBank`` of
    one: its diffuse pyramid is built when an envmap is given or the persistent one changed in place, and calls with
    ``envmap=None`` reuse it (the same image, fewer launches).  ``new_scene=True`` renders build it per call, as before.

    Extra keywords: ``footprint_S`` (Gauss-Legendre sub-normals per cell and axis; None = chosen from the roughness of
    each call, which costs one device-to-host read of z) and ``alpha_min`` (None = max(1e-3, 1.25*pi/He)).  ``spp`` and
    ``denoise`` are kept as attributes because datasets derive cache paths from them
    (dataset/parametricrefmap.py:135-139) but the image is noise free and needs no denoiser.
    """

    def __init__(self, refmap_res: int, spp: int = 1024, envmap_size: tuple = (1000, 2000), denoise: str = None,
                 return_normal: bool = False, return_depth: bool = False, init_view_from: List[float] = [0, 0, 1.1],
                 brdf_param_names: List[str] = None, footprint_S: Optional[int] = None,
                 alpha_min: Optional[float] = None, device="cuda") -> None:
        if denoise:
            assert denoise in ["simple", "informative"], f"{denoise} denoise mode isn't supported"
        self.refmap_res = refmap_res
        self.image_size = (refmap_res, refmap_res)
        self.spp = spp
        self.envmap_size = tuple(envmap_size)
        self.denoise = denoise
        self.return_normal = return_normal
        self.return_depth = return_depth
        self.brdf_param_names = brdf_param_names
        self.footprint_S = footprint_S
        self.alpha_min = alpha_min
        self.device = torch.device(device)
        # persistent-scene state (mitsuba3_utils.py:229-243): envmap, sensor transform, flip, BSDF parameters
        self._envmap: Optional[torch.Tensor] = None
        # the persistent envmap as a bank of one: its diffuse pyramid is built when the map is set or changed in place
        # (identity and version counter of _envmap), not on every call
        self._bank: Optional[EnvmapBank] = None
        self._bank_src: Optional[torch.Tensor] = None
        self._bank_version = -1
        self._view = torch.tensor(init_view_from, dtype=torch.float32)
        self._flip = False
        self._bsdf = torch.tensor(_SCENE_DEFAULTS, dtype=torch.float32)
        # scene_dict["sensor"] is shared by every new_scene render (shallow copy at mitsuba3_utils.py:389)
        self._new_scene_view = self._view.clone()
        self._new_scene_flip = False

    # ------------------------------------------------------------------------------------------------------------
    def _film_res(self, sensor) -> int:
        if isinstance(sensor, int):
            return self.refmap_res
        for attr in ("film_size", "size"):
            v = getattr(sensor, attr, None)
            if v is not None:
                v = v() if callable(v) else v
                return int(v[0])
        if isinstance(sensor, dict) and "film" in sensor:
            return int(sensor["film"]["height"])
        film = getattr(sensor, "film", None)
        if film is not None:
            size = film().size() if callable(film) else film.size()
            return int(size[1])
        raise TypeError(f"sensor {sensor!r}: expected an index or an object carrying a film size")

    def _compose_z6(self, z: torch.Tensor, names: Sequence[str], base: torch.Tensor) -> torch.Tensor:
        """``base`` with the named slots overridden by z, clipped to [0,1] (utils/mitsuba3_utils.py:237-242)."""
        slots = _slots(names)
        z = z.detach().reshape(-1).float().to(self.device)
        if len(slots) > z.numel():
            raise IndexError("z has fewer entries than brdf_param_names")
        z6 = base.clone()
        z6[slots] = z[:len(slots)].clip(0, 1)
        return z6

    def rendering(self, z: torch.Tensor, brdf_param_names: List[str], envmap: torch.Tensor = None,
                  view_from: torch.Tensor = None, flip: bool = None, sensor=0, spp: int = 0, new_scene: bool = False,
                  channel_first: bool = False):
        """One refmap, [res,res,3] or [3,res,res] fp32 CUDA (utils/mitsuba3_utils.py:411-430)."""
        if envmap is not None:
            assert isinstance(envmap, torch.Tensor) and envmap.dim() == 3 and not torch.isnan(envmap[0, 0, 0]), \
                f"envmap [{envmap.shape}]"
        names = brdf_param_names or self.brdf_param_names
        if names is None:
            raise TypeError("brdf_param_names is None and no default was given to the constructor")
        if new_scene:
            if envmap is None:
                raise AttributeError("new_scene=True needs an envmap ('NoneType' object has no attribute 'cuda')")
            env = envmap.to(self.device, _env_dtype(envmap))
            if view_from is not None:
                self._new_scene_view = torch.as_tensor(view_from, dtype=torch.float32).detach().cpu()
            if flip is not None:
                self._new_scene_flip = bool(flip)
            view, do_flip = self._new_scene_view, self._new_scene_flip
            z6 = self._compose_z6(z, names, torch.tensor(_SCENE_DEFAULTS, device=self.device))
        else:
            if envmap is not None:
                self._envmap = envmap.to(self.device, _env_dtype(envmap))
                self._bank = None
            if view_from is not None:
                self._view = torch.as_tensor(view_from, dtype=torch.float32).detach().cpu()
            if flip is not None:
                self._flip = bool(flip)
            if self._envmap is None:
                # the reference would render its initial all-zero bitmap (mitsuba3_utils.py:112)
                self._envmap = torch.zeros(*self.envmap_size, 3, device=self.device)
            env, view, do_flip = self._persistent_bank(), self._view, self._flip
            # parameters that are not named keep their last value in the persistent scene
            self._bsdf = z6 = self._compose_z6(z, names, self._bsdf.to(self.device))
        res = self._film_res(sensor)
        S = self.footprint_S  # None: chosen on the device from the roughness (no host read of z)
        img = render_batch(env if isinstance(env, EnvmapBank) else env[None], z6[None], view[None].to(self.device),
                           flip=torch.tensor([do_flip], device=self.device), res=res, footprint_S=S,
                           alpha_min=self.alpha_min or 0.0, channel_first=channel_first)[0]
        if not self.return_normal and not self.return_depth:
            return img
        outputs = [img]
        if self.return_normal:
            outputs.append(self._normal_aov(res, do_flip, channel_first))
        if self.return_depth:
            outputs.append(self._depth_aov(res, channel_first))
        return outputs

    def _persistent_bank(self) -> EnvmapBank:
        """The bank of the persistent envmap, rebuilt when the envmap was replaced or changed in place."""
        env = self._envmap
        if self._bank is None or self._bank_src is not env or self._bank_version != env._version:
            self._bank = EnvmapBank(env[None])
            self._bank_src, self._bank_version = env, env._version
        return self._bank

    # analytic AOVs of the sphere seen by the refmap sensor (cell centres), mitsuba3_utils.py:199-214
    def _normal_aov(self, res, do_flip, channel_first):
        t = (torch.arange(res, device=self.device) + 0.5) * (torch.pi / res)
        th, ph = torch.meshgrid(t, t, indexing="ij")
        right = -torch.sin(th) * torch.cos(ph) * (-1.0 if do_flip else 1.0)
        n = torch.stack([right, torch.cos(th), torch.sin(th) * torch.sin(ph)], -1)  # [right, up, backward]
        return n.permute(2, 0, 1) if channel_first else n

    def _depth_aov(self, res, channel_first):
        t = (torch.arange(res, device=self.device) + 0.5) * (torch.pi / res)
        th, ph = torch.meshgrid(t, t, indexing="ij")
        depth = 1.1 - torch.sin(th) * torch.sin(ph)
        return depth[None] if channel_first else depth[..., None]
