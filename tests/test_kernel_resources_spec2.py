"""Register and stack budgets of the default specular pass instances (CPU: reads the built library with cuobjdump).

tree_spec_pass2_kernel<P> and its fp16 twin tree_spec_pass2_kernel_h<P> are launched with the grid rule of
tree_spec_pass_kernel<P>, so they have to fit its budget: 80 registers and the 32-byte frame of the sinf / sincosf slow
path, for 3 CTAs of 256 threads per SM (SPEC_MINB in drmnet_b200/csrc/render_tree.cu).
"""
import re

import pytest

from test_kernel_resources_half import FRAME, REGS, resources


def spec2_passes():
    res = {}
    for name, rs in resources().items():
        m = re.fullmatch(r"_ZN3drm2\d(tree_spec_pass2_kernel(?:_h)?)ILi(\d)EEEvNS_8TreeArgsE", name)
        if m:
            res[(m.group(1), int(m.group(2)))] = rs
    return res


def test_every_lattice_has_both_instances():
    assert sorted(spec2_passes()) == [(k, p) for k in ("tree_spec_pass2_kernel", "tree_spec_pass2_kernel_h")
                                      for p in range(5)]


@pytest.mark.parametrize("kernel", ["tree_spec_pass2_kernel", "tree_spec_pass2_kernel_h"])
@pytest.mark.parametrize("p", range(5))
def test_spec_pass2_fits_its_occupancy(kernel, p):
    reg, stack = spec2_passes()[(kernel, p)]
    assert reg <= REGS, f"{kernel}<{p}>: {reg} registers, 80 allow 3 CTAs/SM"
    assert stack <= FRAME, f"{kernel}<{p}>: {stack}-byte stack frame (spills?)"
