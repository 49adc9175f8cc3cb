"""CPU tests of the boundary: the C-ABI library builds, loads and exports every symbol include/stc_b200.h
declares; host-only queries work; the Python cell mirrors the reference's surface and refuses to run
without CUDA (no fallback).  No kernel is launched here."""
import ctypes
import os
import re
import sys

import pytest
import torch

import stc_gnn_b200 as S
from stc_gnn_b200 import _lib
from tests.helpers import GOLDEN, find_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = find_reference()


def header_functions():
    src = open(os.path.join(ROOT, "include", "stc_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(stc_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = header_functions()
    assert set(names) == set(_lib.EXPORTED), (names, _lib.EXPORTED)
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} not exported"
    assert lib.stc_abi_version() == _lib.ABI_VERSION


def test_buffer_size_queries_are_host_only():
    lib = _lib.load()
    d = _lib.StcDims(32, 100, 5, 16, 16, 2, 2, 0, 1)
    saved, scratch = lib.stc_cell_saved_bytes(d), lib.stc_cell_bwd_scratch_bytes(d)
    R = 32 * 100 * 5
    assert saved >= 4 * R * (3 * 16 + 2 * 16 + 16 + 16) and scratch >= 4 * R * 32
    bad = _lib.StcDims(1, 0, 5, 1, 16, 2, 2, 0, 1)
    assert lib.stc_cell_saved_bytes(bad) == 0
    assert b"bad dims" in lib.stc_last_error()


@pytest.mark.parametrize("shape", [(32, 100, 5, 16, 16, 2, 2), (2, 4096, 16, 64, 64, 2, 2), (2, 65536, 8, 64, 64, 4, 2), (3, 7, 3, 1, 4, 1, 1)])
def test_region_layouts_are_host_only_and_consistent(shape):
    """The staged (row-partitioned) path addresses regions of `saved` / `scratch` by these offsets: every region must
    lie inside its buffer, be 256-byte aligned, and leave room for its Ks (or Ks-1) spatial terms before the next one."""
    B, N, C, Din, h, Ks, Kc = shape
    lib = _lib.load()
    d = _lib.StcDims(B, N, C, Din, h, Ks, Kc, 0, 1)
    R = B * N * C
    saved_floats, scratch_floats = lib.stc_cell_saved_bytes(d) // 4, lib.stc_cell_bwd_scratch_bytes(d) // 4
    sv, sc = _lib.saved_layout(d), _lib.scratch_layout(d)
    need_sv = dict(u=R * h, r=R * h, c=R * h, Yr=Ks * R * h, Yx=(Ks - 1) * R * Din, Yh=(Ks - 1) * R * h, Q=Kc * C * C,
                   Pg=R * (Kc - 1) * 2 * h, Pc=R * (Kc - 1) * h)
    need_sc = dict(dYr=Ks * R * h, dYx=(Ks - 1) * R * Din, dYh=(Ks - 1) * R * h)
    for lay, need, total in ((sv, need_sv, saved_floats), (sc, need_sc, scratch_floats)):
        spans = sorted((lay[k], lay[k] + need[k], k) for k in need)
        for (a0, a1, ka), (b0, _, kb) in zip(spans, spans[1:]):
            assert a1 <= b0, f"{ka} overlaps {kb}"
        for a0, a1, k in spans:
            assert a0 % 64 == 0 and a1 <= total, (k, a0, a1, total)
    import ctypes
    small = (ctypes.c_int64 * 2)()
    assert lib.stc_cell_bwd_scratch_layout(d, small, 2) < 0 and b"need room" in lib.stc_last_error()
    assert lib.stc_cell_bwd_stage(d, 7, *([None] * 2), 0, *([None] * 11), 0, None, 0, None, 0, None) < 0   # NULLs: rejected on the host


def test_cell_surface_matches_reference_contract():
    cell = S.STC_Cell(100, 5, 2, 2, 1, 16)
    sd = cell.state_dict()
    assert list(sd.keys()) == ["gates.W", "gates.b", "candi.W", "candi.b"]
    assert tuple(sd["gates.W"].shape) == (17 * 4, 32) and tuple(sd["candi.W"].shape) == (17 * 4, 16)
    assert float(sd["gates.b"].abs().sum()) == 0.0
    assert tuple(cell.init_hidden(3).shape) == (3, 100, 5, 16)
    nb = S.STC_Cell(10, 3, 3, 2, 4, 8, use_bias=False)
    assert list(nb.state_dict().keys()) == ["gates.W", "candi.W"]
    with pytest.raises(NotImplementedError):
        S.STC_Cell(10, 3, 2, 2, 1, 4, activation=torch.nn.Tanh)


def test_no_cpu_fallback():
    cell = S.STC_Cell(6, 3, 2, 2, 1, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cell(Gs=torch.zeros(6, 6), Gc=torch.zeros(3, 3), Xt=torch.zeros(2, 6, 3, 1), Ht_1=torch.zeros(2, 6, 3, 4))
    with pytest.raises(AssertionError):
        cell(Gs=torch.zeros(6, 6), Gc=torch.zeros(3, 3), Xt=torch.zeros(6, 3, 1), Ht_1=torch.zeros(2, 6, 3, 4))


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "stc_gnn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text, f"{f} mentions the oracle"


def test_seeded_init_matches_reference_fixture():
    """The reference's encoder + decoder built in fp64 under torch.manual_seed(5) at the config 5 shapes: the sum of
    |W| over every cell (rounded to fp32) that tests/golden/stack_longc.npz stores.  A seeded RecurrentStack draws the
    same weights only when its cells take the reference's construction order, init and shapes."""
    import numpy as np
    z = np.load(os.path.join(GOLDEN, "stack_longc.npz"))
    B, T, N, C, Din, h, Ks, Kc, layers, horizon = (int(v) for v in z["meta"])
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(int(z["weight_seed"]))
        stack = S.RecurrentStack(N, C, Ks, Kc, Din, h, layers, horizon)
    finally:
        torch.set_default_dtype(prev)
    sd = stack.state_dict()
    assert all(float(v.abs().sum()) == 0.0 for k, v in sd.items() if k.endswith(".b"))
    wsum = sum(float(v.float().double().abs().sum()) for k, v in sd.items() if k.endswith(".W"))
    assert abs(wsum - float(z["weight_checksum"])) < 1e-12 * wsum, (wsum, float(z["weight_checksum"]))


@pytest.mark.skipif(REF_DIR is None, reason="needs the live reference (set STC_REF_DIR)")
def test_seeded_init_and_checkpoint_compat_with_live_reference():
    sys.dont_write_bytecode = True
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import STC_GNN as ref
    torch.manual_seed(123)
    a = ref.STC_Cell(20, 4, 3, 2, 2, 8)
    torch.manual_seed(123)
    b = S.STC_Cell(20, 4, 3, 2, 2, 8)
    for (ka, va), (kb, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert ka == kb and torch.equal(va, vb), ka
    b.load_state_dict(a.state_dict(), strict=True)
    # whole-model: rebinding the module global swaps the cell inside STC_Encoder/STC_Decoder only
    try:
        S.install(ref)
        torch.manual_seed(5)
        enc = ref.STC_Encoder(12, 3, 2, 2, 1, 4, 2)
        assert all(isinstance(c, S.STC_Cell) for c in enc.cell_list)
        from stc_gnn_b200.install import uninstall
        uninstall(ref)
        torch.manual_seed(5)
        enc_ref = ref.STC_Encoder(12, 3, 2, 2, 1, 4, 2)
        assert list(enc.state_dict().keys()) == list(enc_ref.state_dict().keys())
        for k in enc.state_dict():
            assert torch.equal(enc.state_dict()[k], enc_ref.state_dict()[k]), k
        enc.load_state_dict(enc_ref.state_dict(), strict=True)
    finally:
        from stc_gnn_b200.install import uninstall
        uninstall(ref)


def test_sliced_loader_yields_the_reference_dataloaders_batches():
    """SURVEY 8f row f4: the loop-hygiene loaders keep the reference's windowing / split and reproduce its DataLoader's
    batches exactly (order, shapes, last partial batch) -- checked against the live reference's own data path."""
    import io
    from contextlib import redirect_stdout
    from tests.helpers import find_reference
    ref = find_reference()
    if ref is None:
        pytest.skip("needs the live reference")
    import sys
    if ref not in sys.path:
        sys.path.insert(0, ref)
    sys.dont_write_bytecode = True
    import Data_Container as dc
    from stc_gnn_b200.install import SlicedLoader, _patch_loop_hygiene
    with redirect_stdout(io.StringIO()):
        data = dc.DataInput(os.path.join(os.path.dirname(ref), "data", "SF-incidents-4h.npz")).load_data()
    data = dict(data, inc=data["inc"][:400])                       # a slice is enough: 388 windows, 6:1:1
    gen = dc.DataGenerator(obs_len=9, pred_len=3, data_split_ratio=(6, 1, 1))
    params = dict(H=10, W=10, C=5, device="cpu", batch_size=32)
    stock = gen.get_data_loader(params=params, data=data)
    undo = _patch_loop_hygiene(dc)
    try:
        fast = gen.get_data_loader(params=params, data=data)
        assert all(isinstance(v, SlicedLoader) for v in fast.values())
    finally:
        undo()
    assert dc.DataGenerator.get_data_loader(gen, params, data)["train"].__class__.__name__ == "DataLoader"   # undone
    for mode in ("train", "validate", "test"):
        a, b = list(stock[mode]), list(fast[mode])
        assert len(a) == len(b) == len(fast[mode])
        for (xa, ya), (xb, yb) in zip(a, b):
            assert torch.equal(xa, xb) and torch.equal(ya, yb)
    assert a[-1][0].shape[0] != 32 or len(stock["test"].dataset) % 32 == 0   # the partial batch is part of the comparison
