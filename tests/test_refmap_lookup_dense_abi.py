"""The dense refmap lookup at the C ABI, on the host: the refusals that come before any CUDA call, and the ctypes binding
against the header.  Host buffers stand in for device pointers: they are never dereferenced, because every refusal
comes first."""
import ctypes
import re
from pathlib import Path

import pytest

from drmnet_b200 import _lib

HEADER = Path(__file__).resolve().parent.parent / "include" / "drmrender.h"


@pytest.fixture(scope="module")
def lib():
    if not _lib.SO_PATH.exists():
        _lib.build()
    return _lib.lib()


def _call(lib, p, refmap=True, normals=True, ns=(786432, 1536, 3, 1), mask=None, B=2, H=512, W=512, C=3, Hr=128,
          Wr=128, out=True, os=(786432, 512, 1, 262144)):
    ns_arr = None if ns is None else (ctypes.c_int64 * 4)(*ns)
    os_arr = None if os is None else (ctypes.c_int64 * 4)(*os)
    return lib.drm_refmap_lookup_dense(p if refmap else None, Hr, Wr, p if normals else None, ns_arr, mask, B, H, W, C,
                                       p if out else None, os_arr, None)


def test_refusals_come_before_any_cuda_call(lib):
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    n0 = lib.drm_launch_count()

    def refused(*words, **kw):
        rc = _call(lib, p, **kw)
        msg = lib.drm_last_error()
        assert rc == _lib.DRM_EINVAL, (kw, rc, msg)
        for w in words:
            assert w.encode() in msg, (kw, msg)
        return msg

    # null pointers (the mask may be NULL: every pixel)
    for name in ("refmap", "normals", "out"):
        refused("null", **{name: False})
    refused("null", ns=None)
    refused("null", os=None)
    # non-positive sizes, named
    for name, value in (("B", 0), ("H", -3), ("W", 0), ("Hr", 0), ("Wr", -1)):
        refused(f"{name}={value}", **{name: value})
    # channels
    for C in (0, 5, -1):
        refused(f"C={C}", C=C)
    # negative strides, named by position and value
    refused("normals_strides[2] = -3", ns=(786432, 1536, -3, 1))
    refused("out_strides[0] = -1", os=(-1, 512, 1, 262144))
    refused("out_strides[3] = -7", os=(786432, 512, 1, -7))
    # pixel indices of one image are 32-bit
    refused("2147483648", H=65536, W=32768)
    with pytest.raises(ValueError, match="C=5"):
        _lib.check(_call(lib, p, C=5))
    assert lib.drm_launch_count() == n0


def _header_params(name):
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    m = re.search(r"int\s+" + name + r"\s*\((.*?)\)\s*;", text, flags=re.S)
    assert m, name
    return [" ".join(a.split()) for a in m.group(1).split(",")]


def _ctype(param):
    """The ctypes type a header parameter takes in drmnet_b200/_lib.py."""
    if re.search(r"int64_t\s+\w+\[4\]$", param):
        return ctypes.POINTER(ctypes.c_int64)
    if "*" in param:
        return ctypes.c_void_p
    kind = param.rsplit(" ", 1)[0].replace("const ", "")
    return {"int": ctypes.c_int, "float": ctypes.c_float, "int64_t": ctypes.c_int64, "size_t": ctypes.c_size_t}[kind]


def test_binding_matches_the_header(lib):
    params = _header_params("drm_refmap_lookup_dense")
    assert len(params) == 13, params
    assert lib.drm_refmap_lookup_dense.argtypes == [_ctype(a) for a in params]
    assert lib.drm_refmap_lookup_dense.restype is ctypes.c_int
    assert "drm_refmap_lookup_dense" in _lib.EXPORTED_SYMBOLS


def test_python_entries_refuse_host_tensors():
    """The Python entries name the missing CUDA path before any device work."""
    torch = pytest.importorskip("torch")
    from drmnet_b200.callers import refmap_lookup_images
    with pytest.raises(RuntimeError, match="no CPU path"):
        refmap_lookup_images(torch.zeros(1, 3, 8, 8), torch.zeros(1, 3, 4, 4), channel_first=True)
