"""CPU tests of the shared-terms roll-out: the pairing plan of RecurrentStack (stack.share_plan) and the C ABI of the
cell pair that takes supplied terms and folds adjoints (stc_cell_fwd_x / stc_cell_bwd_x).  No kernel is launched."""
import os
import re

import pytest

from stc_gnn_b200 import _lib
from stc_gnn_b200.stack import share_plan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sf_plan():
    """SF shape (2 layers, T = 9, horizon 3): 8 encoder pairs, the encoder-to-decoder pair, 5 decoder pairs, 2 zeros."""
    p = share_plan(2, 9, 3)
    enc = [((("enc", 0, t + 1), "h"), (("enc", 1, t), "x")) for t in range(8)]
    dec = [((("enc", 1, 8), "x"), (("dec", 0, 0), "h")),
           ((("dec", 0, 0), "x"), (("dec", 1, 0), "h")),
           ((("dec", 1, 0), "x"), (("dec", 0, 1), "h")),
           ((("dec", 0, 1), "x"), (("dec", 1, 1), "h")),
           ((("dec", 1, 1), "x"), (("dec", 0, 2), "h")),
           ((("dec", 0, 2), "x"), (("dec", 1, 2), "h"))]
    assert p["pairs"] == enc + dec
    assert len(p["pairs"]) == 14
    assert p["zero"] == [(("enc", 0, 0), "h"), (("enc", 1, 0), "h")]


def test_horizon_zero_and_one():
    p0 = share_plan(2, 4, 0)
    assert p0["pairs"] == [((("enc", 0, t + 1), "h"), (("enc", 1, t), "x")) for t in range(3)]
    p1 = share_plan(2, 4, 1)
    assert p1["pairs"] == p0["pairs"] + [((("enc", 1, 3), "x"), (("dec", 0, 0), "h")),
                                         ((("dec", 0, 0), "x"), (("dec", 1, 0), "h"))]
    assert p0["zero"] == p1["zero"] == [(("enc", 0, 0), "h"), (("enc", 1, 0), "h")]


def test_one_layer_shares_nothing():
    """One layer: each encoder state has one reader, and the decoder reads its state as Xt and as H in the same cell."""
    for horizon in (0, 1, 3):
        p = share_plan(1, 5, horizon)
        assert p["pairs"] == []
        assert p["zero"] == [(("enc", 0, 0), "h")]


def test_single_timestep():
    p = share_plan(2, 1, 2)
    assert p["pairs"] == [((("enc", 1, 0), "x"), (("dec", 0, 0), "h")),
                          ((("dec", 0, 0), "x"), (("dec", 1, 0), "h")),
                          ((("dec", 1, 0), "x"), (("dec", 0, 1), "h")),
                          ((("dec", 0, 1), "x"), (("dec", 1, 1), "h"))]
    assert share_plan(2, 1, 0)["pairs"] == []


def test_three_layers_middle_cell_gives_both_sides():
    """With three layers the middle layer's last encoder cell is the first reader of two states: it gives both sides."""
    p = share_plan(3, 2, 1)
    producers = [pr for pr, _ in p["pairs"]]
    assert (("enc", 1, 1), "x") in producers and (("enc", 1, 1), "h") in producers
    assert len(p["zero"]) == 3


@pytest.mark.parametrize("layers,T,horizon", [(1, 1, 0), (1, 3, 2), (2, 1, 0), (2, 9, 3), (3, 4, 2), (4, 2, 5)])
def test_plan_invariants(layers, T, horizon):
    """Every consumer side takes one producer; a producer runs before its consumer; no cell gives and takes one side."""
    p = share_plan(layers, T, horizon)
    order = [("enc", l, t) for l in range(layers) for t in range(T)] + \
            [("dec", l, s) for s in range(horizon) for l in range(layers)]
    rank = {c: i for i, c in enumerate(order)}
    consumers = [c for _, c in p["pairs"]]
    assert len(set(consumers)) == len(consumers)
    producers = [pr for pr, _ in p["pairs"]]
    assert len(set(producers)) == len(producers)
    assert not set(producers) & set(consumers)
    assert not set(p["zero"]) & (set(producers) | set(consumers))
    for (pc, _), (cc, _) in p["pairs"]:
        assert rank[pc] < rank[cc]
    # every hidden state read twice by two different cells is shared: (layers - 1) * T encoder-internal states, plus
    # the hand-over to and the states inside the decoder when it runs
    expected = (layers - 1) * (T - 1) if layers > 1 else 0
    if horizon and layers > 1:
        expected += layers * horizon
    assert len(p["pairs"]) == expected


def _prototype_params(name):
    src = open(os.path.join(ROOT, "include", "stc_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^)]*)\)\s*;", src)
    assert m, name
    return [a.strip() for a in m.group(1).split(",")]


def test_abi_of_the_shared_terms_pair():
    lib = _lib.load()
    assert _lib.ABI_VERSION == 7 and lib.stc_abi_version() == 7
    fwd, bwd = _prototype_params("stc_cell_fwd_x"), _prototype_params("stc_cell_bwd_x")
    assert [a.split()[-1].lstrip("*") for a in fwd[-3:]] == ["yx_terms", "yh_terms", "stream"]
    assert [a.split()[-1].lstrip("*") for a in bwd[-7:]] == ["yx_terms", "dyx_terms_out", "dyx_fold", "yh_terms",
                                                             "dyh_terms_out", "dyh_fold", "stream"]
    assert len(lib.stc_cell_fwd_x.argtypes) == len(fwd)
    assert len(lib.stc_cell_bwd_x.argtypes) == len(bwd)
