"""Register and stack budgets of the fp16-envmap specular passes (CPU: reads the built library with cuobjdump).

tree_spec_pass_kernel_h<P> is tree_spec_pass_kernel<P> reading fp16 texels.  It is launched with the same grid rule,
so it has to fit the same budget as its fp32 twin: 80 registers and the 32-byte frame of the sinf / sincosf slow path,
for 3 CTAs of 256 threads per SM (SPEC_MINB in drmnet_b200/csrc/render_tree.cu).
"""
import re
import shutil
import subprocess
from pathlib import Path

import pytest

SO = Path(__file__).resolve().parent.parent / "drmnet_b200" / "libdrmrender.so"
REGS, FRAME = 80, 32


def resources():
    exe = shutil.which("cuobjdump")
    if exe is None and Path("/usr/local/cuda/bin/cuobjdump").exists():
        exe = "/usr/local/cuda/bin/cuobjdump"
    if exe is None or not SO.exists():
        pytest.skip("needs cuobjdump and the built drmnet_b200/libdrmrender.so")
    text = subprocess.run([exe, "-res-usage", str(SO)], capture_output=True, text=True, check=True).stdout
    return {m.group(1): (int(m.group(2)), int(m.group(3)))
            for m in re.finditer(r"Function (\w+):\s*REG:(\d+) STACK:(\d+)", text)}


def half_spec_passes():
    res = {}
    for name, rs in resources().items():
        m = re.fullmatch(r"_ZN3drm23tree_spec_pass_kernel_hILi(\d)EEEvNS_8TreeArgsE", name)
        if m:
            res[int(m.group(1))] = rs
    return res


def test_every_lattice_has_its_fp16_instance():
    assert sorted(half_spec_passes()) == [0, 1, 2, 3, 4]


def test_fp16_diffuse_pass_and_pyramid_builds_exist():
    names = resources()
    for name in ("_ZN3drm18tree_diff_kernel_hENS_8TreeArgsE",
                 "_ZN3drm24pyr_from_texels_kernel_hILb0EEEvNS_8TreeArgsEiP6float4",
                 "_ZN3drm24pyr_from_texels_kernel_hILb1EEEvNS_8TreeArgsEiP6float4"):
        assert name in names, name


@pytest.mark.parametrize("p", range(5))
def test_fp16_spec_pass_fits_its_occupancy(p):
    reg, stack = half_spec_passes()[p]
    assert reg <= REGS, f"tree_spec_pass_kernel_h<{p}>: {reg} registers, 80 allow 3 CTAs/SM"
    assert stack <= FRAME, f"tree_spec_pass_kernel_h<{p}>: {stack}-byte stack frame (spills?)"
