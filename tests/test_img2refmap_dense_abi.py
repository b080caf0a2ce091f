"""The dense image -> refmap scatter at the C ABI, on the host: workspace sizes and the refusals that come before any
CUDA call.  Host buffers stand in for device pointers: they are never dereferenced, because every refusal comes first."""
import ctypes
import math

import pytest

from drmnet_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    if not _lib.SO_PATH.exists():
        _lib.build()
    return _lib.lib()


THR = math.pi / 128 / 2


def test_workspace_bytes(lib):
    # 0 for the sizes the entry refuses
    for B, H, W, res, thr in ((0, 8, 8, 16, THR), (1, 0, 8, 16, THR), (1, 8, -1, 16, THR), (1, 8, 8, 0, THR),
                              (1, 8, 8, 16, -1.0), (1, 8, 8, 16, float("nan")), (257, 512, 512, 16, THR)):
        assert lib.drm_img2refmap_dense_workspace_bytes(B, H, W, res, thr) == 0, (B, H, W, res, thr)
    assert lib.drm_img2refmap_dense_workspace_bytes(256, 512, 512, 16, THR) > 0  # exactly 2^26 pixels
    # the compacted entry's workspace at total_n = B*H*W, monotone in B*H*W
    sizes = []
    for B, H, W in ((1, 64, 64), (2, 64, 64), (1, 128, 128), (3, 128, 100), (64, 512, 512)):
        n = lib.drm_img2refmap_dense_workspace_bytes(B, H, W, 128, THR)
        assert n == lib.drm_img2refmap_workspace_bytes(B * H * W, B, 128, THR)
        sizes.append((B * H * W, B, n))
    for (n0, b0, s0), (n1, b1, s1) in zip(sizes, sizes[1:]):
        if n1 >= n0 and b1 >= b0:
            assert s1 >= s0
    for H in (16, 32, 64, 128):
        assert (lib.drm_img2refmap_dense_workspace_bytes(4, H, 64, 64, THR)
                < lib.drm_img2refmap_dense_workspace_bytes(4, 2 * H, 64, 64, THR))


def _call(lib, p, need, colors=True, normals=True, cs=(49152, 384, 3, 1), ns=(49152, 384, 3, 1), mask=None, B=2, H=128,
          W=128, C=3, res=32, thr=THR, reduce=0, refmap=True, refmask=True, ws=True, ws_bytes=None):
    cs_arr = None if cs is None else (ctypes.c_int64 * 4)(*cs)
    ns_arr = None if ns is None else (ctypes.c_int64 * 4)(*ns)
    return lib.drm_img2refmap_dense(p if colors else None, cs_arr, p if normals else None, ns_arr, mask, B, H, W, C, res,
                                    thr, 0, reduce, p if refmap else None, p if refmask else None, None, None,
                                    p if ws else None, need if ws_bytes is None else ws_bytes, None)


def test_refusals_come_before_any_cuda_call(lib):
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    need = lib.drm_img2refmap_dense_workspace_bytes(2, 128, 128, 32, THR)
    assert need > 64
    n0 = lib.drm_launch_count()

    def refused(code=_lib.DRM_EINVAL, *words, **kw):
        rc = _call(lib, p, need, **kw)
        msg = lib.drm_last_error()
        assert rc == code, (kw, rc, msg)
        for w in words:
            assert w.encode() in msg, (kw, msg)
        return msg

    # null pointers (the mask may be NULL: every pixel)
    for name in ("colors", "normals", "refmap", "refmask"):
        refused(_lib.DRM_EINVAL, "null", **{name: False})
    refused(_lib.DRM_EINVAL, "null", cs=None)
    refused(_lib.DRM_EINVAL, "null", ns=None)
    # non-positive sizes, named
    for name, value in (("B", 0), ("H", -3), ("W", 0), ("res", 0)):
        refused(_lib.DRM_EINVAL, f"{name}={value}", **{name: value})
    # channels
    for C in (0, 5):
        refused(_lib.DRM_EINVAL, f"C={C}", C=C)
    # negative strides, named by position and value
    refused(_lib.DRM_EINVAL, "colors_strides[2] = -3", cs=(49152, 384, -3, 1))
    refused(_lib.DRM_EINVAL, "normals_strides[0] = -1", ns=(-1, 384, 3, 1))
    # more than 2^26 dense pixels in one call, whatever the mask holds
    refused(_lib.DRM_EINVAL, "67371008", B=257, H=512, W=512)
    # the threshold and the reduce mode
    refused(_lib.DRM_EINVAL, "threshold", thr=-0.1)
    refused(_lib.DRM_EINVAL, "reduce_mode 2", reduce=2)
    # a workspace that is missing or too small: the size needed is in the message
    refused(_lib.DRM_EWORKSPACE, str(need), ws_bytes=need - 1)
    refused(_lib.DRM_EWORKSPACE, str(need), ws=False)
    with pytest.raises(_lib.DrmError, match=str(need)):
        _lib.check(_call(lib, p, need, ws_bytes=64))
    with pytest.raises(ValueError, match="C=5"):
        _lib.check(_call(lib, p, need, C=5))
    assert lib.drm_launch_count() == n0


def test_python_entry_checks_like_the_batch_entry():
    """Dtype and device errors of img2refmap_images are those of img2refmap_batch, raised before any device work."""
    torch = pytest.importorskip("torch")
    from drmnet_b200.img2refmap import img2refmap_batch, img2refmap_images
    c = torch.zeros(1, 4, 4, 3)
    for fn, args in ((img2refmap_images, (c, c, None, 16, 0.1)),
                     (img2refmap_batch, (c.view(-1, 3), c.view(-1, 3), torch.tensor([0, 16]), 16, 0.1))):
        with pytest.raises(RuntimeError, match="no CPU path"):
            fn(*args, **({"channel_first": False} if fn is img2refmap_images else {}))
