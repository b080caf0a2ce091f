"""ctypes binding of libdrmrender.so (include/drmrender.h).  Fails loudly when the CUDA library is missing:
there is no CPU or PyTorch fallback for the hot path."""
from __future__ import annotations

import ctypes
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
SO_PATH = PKG / "libdrmrender.so"
_lib = None

DRM_OK, DRM_EINVAL, DRM_EWORKSPACE, DRM_ECUDA, DRM_EUNSUPPORTED = 0, -1, -2, -3, -4


class RenderOptions(ctypes.Structure):
    """DrmRenderOptions of include/drmrender.h: accuracy / cost constants of the hierarchical render."""
    _fields_ = [("kappa", ctypes.c_float), ("rcap", ctypes.c_float), ("rcap_simple", ctypes.c_float),
                ("horizon", ctypes.c_float),
                ("kappa_diffuse", ctypes.c_float), ("horizon_diffuse", ctypes.c_float),
                ("level_scale", ctypes.c_float), ("level_scale0", ctypes.c_float),
                ("pixel_covariance", ctypes.c_int), ("full_second_order", ctypes.c_int), ("alpha_full2", ctypes.c_float), ("hand_over", ctypes.c_float), ("limb_nv", ctypes.c_float),
                ("limb_boost", ctypes.c_float), ("limb_x", ctypes.c_float), ("limb_cells", ctypes.c_float), ("limb_sub", ctypes.c_float), ("limb_hand", ctypes.c_float),
                ("limb_ramp", ctypes.c_float), ("flat_scale", ctypes.c_float), ("footprint_per_render", ctypes.c_void_p), ("collect_stats", ctypes.c_int),
                ("horizon_inner", ctypes.c_float), ("horizon_inner_nv", ctypes.c_float), ("horizon_finest", ctypes.c_float)]


def default_render_options() -> "RenderOptions":
    o = RenderOptions()
    lib().drm_render_default_options(ctypes.byref(o))
    return o


class DrmError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libdrmrender error {code}: {message}")
        self.code = code


def build(verbose: bool = False) -> Path:
    """Compile drmnet_b200/csrc/*.cu for sm_100a into drmnet_b200/libdrmrender.so (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", str(PKG / "csrc")], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:], out.stderr[-4000:])
    if out.returncode != 0:
        raise RuntimeError("building libdrmrender.so failed")
    return SO_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not SO_PATH.exists():
        raise ImportError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a). There is no fallback path.")
    L = ctypes.CDLL(str(SO_PATH))
    vp, i32, i64, f32, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_size_t
    L.drm_version.restype = i32
    L.drm_last_error.restype = ctypes.c_char_p
    L.drm_launch_count.restype = i64
    L.drm_render_workspace_bytes.restype = sz
    L.drm_render_workspace_bytes.argtypes = [i32] * 6
    L.drm_render_refmaps.restype = i32
    L.drm_render_refmaps.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, i32, i32, i32, f32, i32, vp, vp, sz, vp]
    L.drm_render_refmaps_opts.restype = i32
    L.drm_render_refmaps_opts.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, i32, i32, i32, f32, i32, vp, vp, sz, vp,
                                          ctypes.POINTER(RenderOptions)]
    L.drm_render_refmaps_half.restype = i32
    L.drm_render_refmaps_half.argtypes = L.drm_render_refmaps_opts.argtypes
    L.drm_env_pyramid_bytes.restype = sz
    L.drm_env_pyramid_bytes.argtypes = [i32] * 3
    L.drm_env_pyramid_build.restype = i32
    L.drm_env_pyramid_build.argtypes = [vp, i32, i32, i32, i32, vp, i32, vp, sz, vp]
    L.drm_render_prepared_workspace_bytes.restype = sz
    L.drm_render_prepared_workspace_bytes.argtypes = [i32] * 6
    L.drm_render_refmaps_prepared.restype = i32
    L.drm_render_refmaps_prepared.argtypes = [vp, i32, vp, sz, i32, i32, i32, vp, vp, vp, vp, i32, i32, i32, f32, i32,
                                              vp, vp, sz, vp, ctypes.POINTER(RenderOptions)]
    L.drm_render_default_options.restype = None
    L.drm_render_default_options.argtypes = [ctypes.POINTER(RenderOptions)]
    L.drm_render_status.restype = i32
    L.drm_render_status.argtypes = [vp, ctypes.POINTER(ctypes.c_int * 40), vp]
    L.drm_render_flat_workspace_bytes.restype = sz
    L.drm_render_flat_workspace_bytes.argtypes = [i32] * 6
    L.drm_render_refmaps_flat.restype = i32
    L.drm_render_refmaps_flat.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, i32, i32, i32, f32, i32, vp, vp, sz, vp]
    L.drm_img2refmap_workspace_bytes.restype = sz
    L.drm_img2refmap_workspace_bytes.argtypes = [i64, i32, i32, f32]
    L.drm_img2refmap.restype = i32
    L.drm_img2refmap.argtypes = [vp, vp, i32, vp, i64, i32, i32, i32, f32, i32, i32, vp, vp, vp, vp, vp, sz, vp]
    L.drm_img2refmap_status.restype = i32
    L.drm_img2refmap_status.argtypes = [vp, i64, i32, i32, f32, ctypes.POINTER(ctypes.c_int32 * 2), vp]
    L.drm_img2refmap_dense_workspace_bytes.restype = sz
    L.drm_img2refmap_dense_workspace_bytes.argtypes = [i32, i32, i32, i32, f32]
    L.drm_img2refmap_dense.restype = i32
    i64p = ctypes.POINTER(i64)
    L.drm_img2refmap_dense.argtypes = [vp, i64p, vp, i64p, vp, i32, i32, i32, i32, i32, f32, i32, i32, vp, vp, vp, vp, vp,
                                       sz, vp]
    L.drm_refmap_postprocess.restype = i32
    L.drm_refmap_postprocess.argtypes = [vp, i32, i32, i32, f32, i32, vp, vp, vp]
    L.drm_mirmap2envmap.restype = i32
    L.drm_mirmap2envmap.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp]
    L.drm_refmap_lookup.restype = i32
    L.drm_refmap_lookup.argtypes = [vp, vp, vp, i64, i32, i32, i32, i32, vp, vp]
    L.drm_normalized_log.restype = i32
    L.drm_normalized_log.argtypes = [vp, vp, i32, i32, i32, i32, f32, vp, vp, vp, vp]
    L.drm_obsnet_condition.restype = i32
    L.drm_obsnet_condition.argtypes = [vp, vp, i32, i32, i32, i32, f32, f32, vp, vp, vp, vp, vp, vp]
    L.drm_normalized_log_apply.restype = i32
    L.drm_normalized_log_apply.argtypes = [vp, vp, vp, i32, i32, i32, i32, f32, i32, f32, vp, vp]
    L.drm_normals_to_thetaphi.restype = i32
    L.drm_normals_to_thetaphi.argtypes = [vp, i64, vp, vp]
    _lib = L
    return L


def check(code: int) -> None:
    if code != DRM_OK:
        msg = lib().drm_last_error().decode("utf-8", "replace")
        if code == DRM_EINVAL:
            raise ValueError(f"libdrmrender: {msg}")
        raise DrmError(code, msg)


EXPORTED_SYMBOLS = ["drm_version", "drm_last_error", "drm_launch_count", "drm_render_workspace_bytes", "drm_render_refmaps",
                    "drm_render_refmaps_opts", "drm_render_refmaps_half", "drm_render_default_options", "drm_render_status",
                    "drm_env_pyramid_bytes", "drm_env_pyramid_build", "drm_render_prepared_workspace_bytes",
                    "drm_render_refmaps_prepared",
                    "drm_render_flat_workspace_bytes", "drm_render_refmaps_flat",
                    "drm_img2refmap_workspace_bytes", "drm_img2refmap", "drm_img2refmap_status", "drm_normals_to_thetaphi",
                    "drm_img2refmap_dense_workspace_bytes", "drm_img2refmap_dense",
                    "drm_refmap_postprocess", "drm_mirmap2envmap", "drm_refmap_lookup", "drm_normalized_log",
                    "drm_obsnet_condition", "drm_normalized_log_apply"]
