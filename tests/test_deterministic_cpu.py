"""Host-only checks of the deterministic mode's C ABI (stc_deterministic_set, the scratch slots, the workspace of
stc_support_outer_ws).  No kernel is launched; every test leaves the mode off."""
import ctypes

import pytest

from stc_gnn_b200 import _lib

SHAPES = [(32, 100, 5, 16, 16, 2, 2), (2, 4096, 16, 64, 64, 2, 2), (2, 65536, 8, 64, 64, 4, 2), (3, 7, 3, 1, 4, 1, 1)]
# stc_cell_bwd_scratch_bytes and the (dYr, dYx, dYh) offsets of the library before the deterministic mode existed: the
# default layout must stay exactly this
DEFAULT_SCRATCH = {
    (32, 100, 5, 16, 16, 2, 2): (9216256, [1792000, 1280000, 1536000]),
    (2, 4096, 16, 64, 64, 2, 2): (302516224, [58720256, 41943040, 50331648]),
    (2, 65536, 8, 64, 64, 4, 2): (4027580928, [738197504, 335544320, 536870912]),
    (3, 7, 3, 1, 4, 1, 1): (3584, [576, 576, 576]),
}


@pytest.fixture
def lib():
    lib = _lib.load()
    yield lib
    assert lib.stc_deterministic_set(0) == 0
    _lib._DET_SENT = 0


def _layout(lib, d, n):
    offs = (ctypes.c_int64 * n)()
    assert lib.stc_cell_bwd_scratch_layout(d, offs, n) == 0
    return list(offs)


def test_new_exports_present(lib):
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in ("stc_deterministic_set", "stc_support_outer_ws", "stc_support_outer_workspace_bytes"):
        assert name in _lib.EXPORTED and hasattr(raw, name)


@pytest.mark.parametrize("bad", [-1, 2, 7])
def test_set_rejects_other_values(lib, bad):
    assert lib.stc_deterministic_set(bad) == -1
    assert b"stc_deterministic_set" in lib.stc_last_error()
    assert lib.stc_deterministic_set(1) == 0 and lib.stc_deterministic_set(0) == 0


@pytest.mark.parametrize("shape", SHAPES)
def test_scratch_sizes_and_layouts(lib, shape):
    """Off: exactly the default sizes and offsets (the slot offset is the end of the buffer).  On: the default regions
    keep their offsets, the buffer grows, and the slots start after every default region."""
    B, N, C, Din, h, Ks, Kc = shape
    d = _lib.StcDims(B, N, C, Din, h, Ks, Kc, 0, 1)
    saved_off, scratch_off = lib.stc_cell_saved_bytes(d), lib.stc_cell_bwd_scratch_bytes(d)
    lay_off = _layout(lib, d, len(_lib.SCRATCH_REGIONS) + 1)
    assert (scratch_off, lay_off[:3]) == DEFAULT_SCRATCH[shape]
    assert lay_off[:3] == list(_lib.scratch_layout(d).values())
    assert lay_off[3] * 4 == scratch_off
    assert lib.stc_deterministic_set(1) == 0
    saved_on, scratch_on = lib.stc_cell_saved_bytes(d), lib.stc_cell_bwd_scratch_bytes(d)
    lay_on = _layout(lib, d, len(_lib.SCRATCH_REGIONS) + 1)
    assert saved_on == saved_off                      # the forward's buffer does not depend on the mode
    assert lay_on[:3] == lay_off[:3]
    assert lay_on[3] * 4 == scratch_off               # the slots begin where the default buffer ends
    R, P, L = B * N * C, Ks * Kc, Din + h
    assert scratch_on >= scratch_off + 4 * P * L * 2 * h   # at least one dW slot
    assert lib.stc_deterministic_set(0) == 0
    assert lib.stc_cell_bwd_scratch_bytes(d) == scratch_off
    assert R > 0


def test_outer_workspace_is_host_only(lib):
    assert lib.stc_support_outer_workspace_bytes(100, 4096, 80) == 0          # mode off: no slots
    assert lib.stc_deterministic_set(1) == 0
    n = lib.stc_support_outer_workspace_bytes(100, 4096, 80)
    assert n > 0 and n % (4 * 100 * 100) == 0                               # whole N x N slots
    assert lib.stc_support_outer_workspace_bytes(100, 1, 80) == 0            # one sample slice: one writer per element
    assert lib.stc_support_outer_workspace_bytes(0, 4, 80) == 0
    assert lib.stc_support_outer_workspace_bytes(65536, 2, 512) == 0          # one slice of 128 x 128 blocks
    # the plain entry point refuses the mode on the host, naming its sibling
    assert lib.stc_support_outer(100, 4, 80, ctypes.c_void_p(16), 8000, ctypes.c_void_p(16), 1.0,
                                 ctypes.c_void_p(16), None) == -2
    assert b"stc_support_outer_ws" in lib.stc_last_error()
    assert lib.stc_support_outer_ws(100, 4096, 80, ctypes.c_void_p(16), 8000, ctypes.c_void_p(16), 1.0,
                                    ctypes.c_void_p(16), None, 0, None) == -3


def test_python_follows_torch_switch(lib):
    torch = pytest.importorskip("torch")
    was = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        assert _lib.sync_deterministic() is True
        assert lib.stc_support_outer_workspace_bytes(100, 4096, 80) > 0
        torch.use_deterministic_algorithms(False)
        assert _lib.sync_deterministic() is False
        assert lib.stc_support_outer_workspace_bytes(100, 4096, 80) == 0
    finally:
        torch.use_deterministic_algorithms(was)
