"""Register and stack budgets of the specular lattice passes (CPU: reads the built library with cuobjdump).

An instance that runs at 3 CTAs of 256 threads per SM has 80 registers a thread; an edit that pushes it past that makes
ptxas spill to local memory, and the pass slows down without any test failing.  The budgets follow SPEC_MINB in
drmnet_b200/csrc/render_tree.cu.
"""
import re
import shutil
import subprocess
from pathlib import Path

import pytest

SO = Path(__file__).resolve().parent.parent / "drmnet_b200" / "libdrmrender.so"
MINB = {0: 3, 1: 3, 2: 3, 3: 3, 4: 3}  # resident CTAs per SM of tree_spec_pass_kernel<P> (SPEC_MINB)
FRAME = 32  # bytes: the local table of the slow path of sinf / sincosf in make_node, never reached by the item loop


def _cuobjdump():
    exe = shutil.which("cuobjdump")
    if exe is None and Path("/usr/local/cuda/bin/cuobjdump").exists():
        exe = "/usr/local/cuda/bin/cuobjdump"
    return exe


def spec_pass_resources():
    exe = _cuobjdump()
    if exe is None or not SO.exists():
        pytest.skip("needs cuobjdump and the built drmnet_b200/libdrmrender.so")
    text = subprocess.run([exe, "-res-usage", str(SO)], capture_output=True, text=True, check=True).stdout
    res = {}
    for m in re.finditer(r"Function _ZN3drm21tree_spec_pass_kernelILi(\d)EEEvNS_8TreeArgsE:\s*REG:(\d+) STACK:(\d+)", text):
        res[int(m.group(1))] = (int(m.group(2)), int(m.group(3)))
    return res


def test_every_lattice_has_its_instance():
    assert sorted(spec_pass_resources()) == [0, 1, 2, 3, 4]


@pytest.mark.parametrize("p", range(5))
def test_spec_pass_fits_its_occupancy(p):
    reg, stack = spec_pass_resources()[p]
    if MINB[p] >= 3:
        assert reg <= 80, f"tree_spec_pass_kernel<{p}>: {reg} registers, 80 allow 3 CTAs/SM"
        assert stack <= FRAME, f"tree_spec_pass_kernel<{p}>: {stack}-byte stack frame (spills?)"
    else:
        assert reg <= 128, f"tree_spec_pass_kernel<{p}>: {reg} registers, 128 allow 2 CTAs/SM"
