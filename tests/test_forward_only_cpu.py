"""Host-only checks of the forward-only cell calls (stc_cell_fwd_only*, cell.FORWARD_ONLY): the exports, the size and
layout of the smaller workspace, the unchanged training buffers, and which calls take the forward-only form.  No
kernel is launched."""
import ctypes

import pytest
import torch

import stc_gnn_b200 as S
from stc_gnn_b200 import _lib, cell

NEW = ("stc_cell_fwd_only_bytes", "stc_cell_fwd_only_layout", "stc_cell_fwd_only", "stc_cell_fwd_only_stage")
# (B, N, C, Din, h, Ks, Kc): SF at Din = 1 and 16, a wide hidden state (h = 64, Ks = 4: both weight images), the
# general path (h = 6, Kc = 3) and Kc = 1 (no P_1 partials at all)
SHAPES = [(32, 100, 5, 1, 16, 2, 2), (32, 100, 5, 16, 16, 2, 2), (2, 4096, 16, 64, 64, 4, 2), (3, 33, 5, 4, 6, 2, 3),
          (3, 7, 3, 1, 4, 1, 1)]
# stc_cell_saved_bytes and stc_cell_bwd_scratch_bytes of these shapes before the forward-only calls existed
TRAINING_BYTES = {
    (32, 100, 5, 1, 16, 2, 2): (9280256, 7296256),
    (32, 100, 5, 16, 16, 2, 2): (10240256, 9216256),
    (2, 4096, 16, 64, 64, 4, 2): (538445824, 504367104),
    (3, 33, 5, 4, 6, 2, 3): (151808, 123648),
    (3, 7, 3, 1, 4, 1, 1): (4352, 3584),
}


def ru(n):   # every region starts 256-byte aligned
    return (n + 63) // 64 * 64


def fwd_only_layout(lib, d):
    offs = (ctypes.c_int64 * len(_lib.SAVED_REGIONS))()
    assert lib.stc_cell_fwd_only_layout(d, offs, len(offs)) == 0
    return dict(zip(_lib.SAVED_REGIONS, offs))


def test_exports_match_the_header():
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in NEW:
        assert name in _lib.EXPORTED and hasattr(raw, name)
    assert _lib.load().stc_abi_version() == 7


@pytest.mark.parametrize("shape", SHAPES)
def test_workspace_is_the_sum_of_its_regions(shape):
    B, N, C, Din, h, Ks, Kc = shape
    lib = _lib.load()
    d = _lib.StcDims(B, N, C, Din, h, Ks, Kc, 0, 1)
    R = B * N * C
    ws = lib.stc_cell_fwd_only_bytes(d)
    saved = lib.stc_cell_saved_bytes(d)
    lay = fwd_only_layout(lib, d)
    assert [lay[k] for k in ("r", "c", "Pg", "Pc")] == [-1] * 4
    # u, Yr[Ks], Yx[Ks-1], Yh[Ks-1], Q back to back, then the wide-state weight images (the only regions left)
    o = 0
    for name, n in (("u", R * h), ("Yr", Ks * R * h), ("Yx", (Ks - 1) * R * Din), ("Yh", (Ks - 1) * R * h),
                    ("Q", Kc * C * C)):
        assert lay[name] == o, (name, lay)
        o += ru(n)
    # the training buffer is this one plus r, c and the P_1 partials, with the same weight images
    dropped = 2 * ru(R * h) + ru(R * (Kc - 1) * 2 * h) + ru(R * (Kc - 1) * h)
    assert saved - ws == 4 * dropped
    assert ws <= saved and ws >= 4 * o
    if h < 32:   # no wide-state weight image at these widths
        assert ws == 4 * o
    assert lay == _lib.saved_layout(d, fwd_only=True)


@pytest.mark.parametrize("shape", SHAPES)
def test_training_buffers_are_unchanged(shape):
    B, N, C, Din, h, Ks, Kc = shape
    lib = _lib.load()
    d = _lib.StcDims(B, N, C, Din, h, Ks, Kc, 0, 1)
    assert (lib.stc_cell_saved_bytes(d), lib.stc_cell_bwd_scratch_bytes(d)) == TRAINING_BYTES[shape]
    assert -1 not in _lib.saved_layout(d).values()


def test_host_side_argument_checks():
    lib = _lib.load()
    d = _lib.StcDims(2, 10, 5, 1, 16, 2, 2, 0, 1)
    small = (ctypes.c_int64 * 2)()
    assert lib.stc_cell_fwd_only_layout(d, small, 2) == -1 and b"need room" in lib.stc_last_error()
    bad = _lib.StcDims(1, 0, 5, 1, 16, 2, 2, 0, 1)
    assert lib.stc_cell_fwd_only_bytes(bad) == 0
    # NULL arguments and a bad stage are refused before anything touches a device
    assert lib.stc_cell_fwd_only(d, None, *([None] * 2), 0, *([None] * 6), None, 0, None, None, None) == -1
    assert lib.stc_cell_fwd_only_stage(d, 7, *([None] * 2), 0, *([None] * 6), None, 0, None) == -1


def test_forward_only_selection(monkeypatch):
    leaf = torch.zeros(3, requires_grad=True)
    plain = torch.zeros(3)
    monkeypatch.setattr(cell, "FORWARD_ONLY", True)
    assert cell.forward_only(plain, None)                     # nothing requires grad
    assert not cell.forward_only(plain, leaf)                 # a gradient can be asked for
    with torch.no_grad():
        assert cell.forward_only(plain, leaf)
    with torch.inference_mode():
        assert cell.forward_only(plain, leaf)
    monkeypatch.setattr(cell, "FORWARD_ONLY", False)          # the A/B switch keeps the training forward
    with torch.no_grad():
        assert not cell.forward_only(plain)


def test_forward_only_refuses_cpu_tensors_with_the_training_message():
    c = S.STC_Cell(10, 3, 2, 2, 1, 4)
    Gs, Gc = torch.rand(10, 10), torch.rand(3, 3)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        c(Gs, Gc, torch.rand(2, 10, 3, 1), c.init_hidden(2))
