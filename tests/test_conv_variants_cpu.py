"""Host-side checks of tests/test_conv_variants_gpu.py: its variant list is exactly the set of convolution kernels the
built library contains, and its multi-tile sizing gives every multi-tile case at least 3 tiles per CTA on a B200."""
import os
import re
import shutil
import subprocess

import pytest

from tests import test_conv_variants_gpu as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "stc_gnn_b200", "libstc_b200.so")


def _cuobjdump():
    for cand in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if cand and os.path.exists(cand):
            return cand
    return None


def test_variant_list_equals_the_library_instantiations():
    tool = _cuobjdump()
    if not os.path.exists(LIB) or tool is None:
        pytest.skip("library not built or cuobjdump not found")
    out = subprocess.run([tool, "-symbols", LIB], capture_output=True, text=True, check=True).stdout
    mangled = set(re.findall(r"STO_ENTRY\s+(\S+)", out))
    demangled = subprocess.run(["c++filt"], input="\n".join(sorted(mangled)), capture_output=True, text=True,
                               check=True).stdout.splitlines()
    built = {n for n in (V.conv_kernel_name(d) for d in demangled) if n}
    listed = set(V.VARIANTS)
    assert len(listed) == len(V.VARIANTS), "duplicate entries in VARIANTS"
    assert built == listed | set(V.EXCLUDED), (f"in the library but not in the GPU test's list: {sorted(built - listed)}; "
                                               f"listed but not in the library: {sorted(listed - built)}")
    covered = set().union(*(c["kernels"] for c in V.CASES.values()))
    assert covered == listed - set(V.EXCLUDED), f"listed variants no case launches: {sorted(listed - covered)}"
    multi = set().union(*(V.CASES[n]["kernels"] for n in V.MULTI_TILE))
    assert multi == listed - set(V.EXCLUDED), f"variants without a multi-tile case: {sorted(listed - multi)}"


def test_kernel_name_reduction():
    assert V.conv_kernel_name("void stc::tc_conv_bwd_dx_kernel<true, false>(stc::ConvArgs, stc::TcDxPlan)") == \
        "tc_conv_bwd_dx_kernel<true, false>"
    assert V.conv_kernel_name("stc::tc_conv_fwd_big_kernel(stc::ConvArgs, stc::BigPlan, unsigned char const*)") == \
        "tc_conv_fwd_big_kernel"
    assert V.conv_kernel_name("void stc::tc_support_kernel<true>(float const*)") is None
    assert V.conv_kernel_name("stc::tc_big_prep_kernel(float const*, unsigned char*, int)") is None


@pytest.mark.parametrize("name", V.MULTI_TILE)
def test_multi_tile_sizing_on_148_sms(name):
    spec = V.CASES[name]
    sms = 148
    B, node_tiles, dw_tiles = V.multi_tile_batch(spec["N"], spec["C"], sms)
    grid = 2 * sms
    npt = 128 // spec["C"]
    assert (B * spec["N"] + npt - 1) // npt >= 3 * grid and node_tiles >= 3, (B, node_tiles)
    assert (B * spec["N"] * spec["C"] + 63) // 64 >= 3 * grid and dw_tiles >= 3, (B, dw_tiles)
    assert ((B * spec["N"] + npt - 1) // npt) % grid != 0, "the last wave must be partial"
    if spec["N"] % npt:
        assert (B * spec["N"]) % npt != 0, "the last node tile must be ragged"
