"""Envmap banks at the C ABI, on the host: buffer and workspace sizes, the checks that run before any CUDA call, and the
SASS of the kernels that existed before banks (the bank entries reuse them and must leave them as they were)."""
import ctypes
import hashlib
import json
import re
import shutil
import subprocess
from pathlib import Path

import pytest

from drmnet_b200 import _lib

ROOT = Path(__file__).resolve().parent.parent
SASS_GOLDEN = ROOT / "tests" / "golden" / "kernel_sass_v200.json"


@pytest.fixture(scope="module")
def lib():
    if not _lib.SO_PATH.exists():
        _lib.build()
    return _lib.lib()


def diffuse_cells(He, We):
    """Records of one diffuse pyramid: the levels from the first one whose cells reach ~0.03 rad up to <= 256 cells."""
    H, W, levels = [He], [We], 0
    while H[-1] * W[-1] > 256 and levels + 1 < 14:
        H.append((H[-1] + 1) // 2)
        W.append((W[-1] + 1) // 2)
        levels += 1
    base = 0
    while (2 << base) * 3.141592653589793 / He <= 0.03:
        base += 1
    base = min(base, levels)
    return max(sum(H[i] * W[i] for i in range(max(base, 1), levels + 1)), 1)


def test_pyramid_bytes_linear_in_B(lib):
    for He, We in ((1000, 2000), (128, 256), (250, 500)):
        per_map = diffuse_cells(He, We) * 5 * 16
        sizes = [lib.drm_env_pyramid_bytes(B, He, We) for B in (64, 128, 192, 1024)]
        assert sizes[1] - sizes[0] == sizes[2] - sizes[1]
        # records plus one mask int per map, nothing else that grows with B
        assert sizes[1] - sizes[0] == 64 * (per_map + 4)
        assert sizes[3] - sizes[0] == 960 * (per_map + 4)
    assert 3.3e6 < diffuse_cells(1000, 2000) * 80 < 3.5e6
    assert lib.drm_env_pyramid_bytes(0, 1000, 2000) == 0
    assert lib.drm_env_pyramid_bytes(65536, 16, 32) == 0
    assert lib.drm_env_pyramid_bytes(1, 1 << 14, 1 << 14) == 0


def test_prepared_workspace_does_not_grow_with_B(lib):
    for N, res, S in ((64, 128, 0), (1, 128, 1), (200, 256, 4)):
        prep = [lib.drm_render_prepared_workspace_bytes(N, B, 1000, 2000, res, S) for B in (64, 1024, 4096)]
        full = [lib.drm_render_workspace_bytes(N, B, 1000, 2000, res, S) for B in (64, 1024, 4096)]
        assert prep[1] - prep[0] <= 4 * 960 and prep[2] - prep[1] <= 4 * 3072
        # today's workspace carries a diffuse pyramid per map: ~3.4 MB at 2000 x 1000
        per_map = (full[1] - full[0]) / 960
        assert 3.3e6 < per_map < 3.5e6
        assert prep[0] < full[0]
    assert lib.drm_render_prepared_workspace_bytes(1, 1, 1000, 2000, 128, 3) == 0
    assert lib.drm_render_prepared_workspace_bytes(0, 1, 1000, 2000, 128, 1) == 0


def _prepared(lib, env, pyr, pyr_bytes, ws, ws_bytes, S=2, B=1, He=64, We=128, z=None, v=None, out=None):
    return lib.drm_render_refmaps_prepared(env, 0, pyr, pyr_bytes, B, He, We, None, z, v, None, 1, 16, S, 0.0, 1, out,
                                           ws, ws_bytes, None, None)


def test_prepared_render_checks_before_any_device_work(lib):
    """Host buffers stand in for device pointers: they are never dereferenced, because every refusal comes first."""
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    need_pyr = lib.drm_env_pyramid_bytes(1, 64, 128)
    need_ws = lib.drm_render_prepared_workspace_bytes(1, 1, 64, 128, 16, 2)
    assert need_pyr > 64 and need_ws > 64
    # null pointers: envmap, pyramids, z / view / out
    for args in ((None, p), (p, None)):
        rc = _prepared(lib, args[0], args[1], need_pyr, p, need_ws, z=p, v=p, out=p)
        assert rc == _lib.DRM_EINVAL and b"null" in lib.drm_last_error()
    rc = _prepared(lib, p, p, need_pyr, p, need_ws, z=None, v=p, out=p)
    assert rc == _lib.DRM_EINVAL and b"null" in lib.drm_last_error()
    # a pyramid buffer that is too small: the size needed is in the message
    rc = _prepared(lib, p, p, need_pyr - 1, p, need_ws, z=p, v=p, out=p)
    assert rc == _lib.DRM_EINVAL and str(need_pyr).encode() in lib.drm_last_error()
    with pytest.raises(ValueError, match=str(need_pyr)):
        _lib.check(rc)
    # a workspace that is too small, with a pyramid buffer that is large enough
    rc = _prepared(lib, p, p, need_pyr, p, 64, z=p, v=p, out=p)
    assert rc == _lib.DRM_EWORKSPACE and str(need_ws).encode() in lib.drm_last_error()
    # the same size checks as drm_render_refmaps
    rc = _prepared(lib, p, p, need_pyr, p, need_ws, S=3, z=p, v=p, out=p)
    assert rc == _lib.DRM_EINVAL and b"footprint_S" in lib.drm_last_error()
    rc = _prepared(lib, p, p, need_pyr, p, need_ws, B=0, z=p, v=p, out=p)
    assert rc == _lib.DRM_EINVAL


def test_pyramid_build_checks_before_any_device_work(lib):
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    need = lib.drm_env_pyramid_bytes(3, 64, 128)
    rc = lib.drm_env_pyramid_build(None, 0, 3, 64, 128, None, 0, p, need, None)
    assert rc == _lib.DRM_EINVAL and b"null" in lib.drm_last_error()
    rc = lib.drm_env_pyramid_build(p, 1, 3, 64, 128, None, 0, None, need, None)
    assert rc == _lib.DRM_EINVAL and b"null" in lib.drm_last_error()
    for half in (0, 1):
        rc = lib.drm_env_pyramid_build(p, half, 3, 64, 128, None, 0, p, need - 1, None)
        assert rc == _lib.DRM_EINVAL and str(need).encode() in lib.drm_last_error()
    rc = lib.drm_env_pyramid_build(p, 0, 3, 64, 128, p, -1, p, need, None)
    assert rc == _lib.DRM_EINVAL and b"n_ids" in lib.drm_last_error()
    rc = lib.drm_env_pyramid_build(p, 0, 65536, 64, 128, None, 0, p, 1 << 40, None)
    assert rc == _lib.DRM_EINVAL
    # an empty id list is nothing to do: no launch, no CUDA call
    n0 = lib.drm_launch_count()
    assert lib.drm_env_pyramid_build(p, 0, 3, 64, 128, p, 0, p, need, None) == _lib.DRM_OK
    assert lib.drm_launch_count() == n0


def _nvcc_release():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    try:
        text = subprocess.run([exe, "--version"], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.CalledProcessError):
        return None
    m = re.search(r"release [\d.]+, V[\d.]+", text)
    return m.group(0) if m else None


def _sass_by_kernel(so):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    text = subprocess.run([exe, "-sass", str(so)], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if m and cur is not None:
            cur.append(m.group(1))
    return out


def test_existing_kernels_keep_their_sass(lib):
    """Every kernel of the library before banks compiles to the same instructions: the bank entries only add host code
    and one marking kernel around the existing pyramid kernels."""
    golden = json.loads(SASS_GOLDEN.read_text())
    if not (shutil.which("cuobjdump") or Path("/usr/local/cuda/bin/cuobjdump").exists()):
        pytest.skip("needs cuobjdump")
    release = _nvcc_release()
    if release != golden["compiler"]:
        pytest.skip(f"recorded with nvcc {golden['compiler']}, this toolkit is {release}")
    sass = _sass_by_kernel(_lib.SO_PATH)
    for name, want in golden["kernels"].items():
        assert name in sass, f"{name} is missing"
        got = sass[name]
        assert len(got) == want["instructions"], f"{name}: {len(got)} instructions, {want['instructions']} recorded"
        assert hashlib.sha256("\n".join(got).encode()).hexdigest() == want["sha256"], f"{name}: instructions differ"
