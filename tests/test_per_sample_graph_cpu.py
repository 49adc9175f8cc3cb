"""Per-sample spatial graphs, CPU side: the ABI constants of the new support kind, and the fp64 per-sample restatements
(tests/per_sample_oracle.py) against the single-sample oracles applied to each sample and stacked."""
import ctypes
import os
import re

import pytest
import torch

from oracle import stc_oracle as O
from stc_gnn_b200 import _lib
from tests import per_sample_oracle as PS
from tests import sparse_mgp_oracle as M
from tests.helpers import random_case
from tests.learned_csr_oracle import stc_cell_edge_grad

HEADER = os.path.join(os.path.dirname(__file__), "..", "include", "stc_b200.h")


def test_header_and_binding_have_the_per_sample_kind():
    text = open(HEADER).read()
    m = re.search(r"enum \{ STC_SUPPORT_DENSE = 0, STC_SUPPORT_CSR = 1, STC_SUPPORT_CSR_PER_SAMPLE = (\d+) \};", text)
    assert m and int(m.group(1)) == 2 == _lib.SUPPORT_CSR_PER_SAMPLE
    assert (_lib.SUPPORT_DENSE, _lib.SUPPORT_CSR) == (0, 1)
    assert re.search(r"#define STC_ABI_VERSION 7\b", text) and _lib.ABI_VERSION == 7
    for name in ("stc_pair_scores_csr_batched", "stc_edge_softmax_fwd_batched", "stc_edge_softmax_bwd_batched"):
        assert name in _lib.EXPORTED and re.search(rf"\bint {name}\(", text), name


def test_support_struct_layout_is_unchanged():
    S = _lib.StcSupport
    offs = [(n, getattr(S, n).offset) for n, _ in S._fields_]
    assert offs == [("kind", 0), ("nnz", 8), ("vals", 16), ("rowptr", 24), ("col", 32), ("t_vals", 40),
                    ("t_rowptr", 48), ("t_col", 56)]
    assert ctypes.sizeof(S) == 64


def pattern(N, deg, seed):
    """A pattern with empty rows, self-loops and explicit zero values in every sample."""
    rowptr, col = M.random_pattern(N, deg, seed, empty_every=6, self_loop_every=3)
    assert (rowptr[1:] == rowptr[:-1]).any() and (M.edge_rows(rowptr) == col.long()).any()
    return rowptr, col


def per_sample_values(B, nnz, deg, seed):
    g = torch.Generator().manual_seed(seed)
    vals = ((torch.rand(B, nnz, generator=g) + 0.5) / deg).double()
    vals[torch.rand(B, nnz, generator=g) < 0.2] = 0.0
    return vals


@pytest.mark.parametrize("Ks", [1, 2, 3, 4])
@pytest.mark.parametrize("Kc", [1, 2, 3])
def test_per_sample_cell_is_the_single_sample_oracle_stacked(Ks, Kc):
    B, N, C, Din, h = 3, 19, 3, 2, 4
    rowptr, col = pattern(N, 4, seed=Ks * 5 + Kc)
    vals = per_sample_values(B, col.numel(), 4, seed=Ks + 7 * Kc)
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=11 * Ks + Kc)
    Hn, g = PS.cell_with_grads(t, rowptr, col, vals, Ks, Kc)
    sum_keys = ("dWg", "dWc", "dbg", "dbc", "dGc")
    acc = {k: 0.0 for k in sum_keys}
    for b in range(B):
        sl = slice(b, b + 1)
        Gs_b = torch.sparse_csr_tensor(rowptr.long(), col.long(), vals[b], size=(N, N))
        tb = {k: (t[k][sl] if k in ("Xt", "H", "dHn") else t[k]) for k in t}
        names = ["Gc", "Xt", "H", "Wg", "Wc", "bg", "bc"]
        v = {k: tb[k].double().clone().requires_grad_(True) for k in names}
        Hb = O.stc_cell(Gs_b.to_dense(), v["Gc"], v["Xt"], v["H"], v["Wg"], v["bg"], v["Wc"], v["bc"], Ks, Kc)
        Hb.backward(tb["dHn"].double())
        torch.testing.assert_close(Hn[sl], Hb.detach(), rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(g["dXt"][sl], v["Xt"].grad, rtol=1e-10, atol=1e-12)
        torch.testing.assert_close(g["dH"][sl], v["H"].grad, rtol=1e-10, atol=1e-12)
        for k, name in (("Wg", "dWg"), ("Wc", "dWc"), ("bg", "dbg"), ("bc", "dbc"), ("Gc", "dGc")):
            acc[name] = acc[name] + (v[k].grad if v[k].grad is not None else torch.zeros_like(v[k]))
        dv = stc_cell_edge_grad(Gs_b, tb["Gc"], tb["Xt"], tb["H"], tb["Wg"], tb["bg"], tb["Wc"], tb["bc"], Ks, Kc,
                                tb["dHn"])
        torch.testing.assert_close(g["dvals"][b], dv, rtol=1e-10, atol=1e-12)
        if Ks > 1:
            assert float(g["dvals"][b][vals[b] == 0].abs().max()) > 0.0, "an edge stored as 0 still gets a gradient"
    for name in sum_keys:
        torch.testing.assert_close(g[name], acc[name], rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("pat", ["random", "complete"])
def test_per_sample_generator_is_the_sparse_generator_on_each_window(pat):
    B, T, N, C, hg = 3, 4, 13, 3, 5
    rowptr, col = pattern(N, 5, seed=3) if pat == "random" else M.complete_pattern(N)
    g = torch.Generator().manual_seed(5)
    X = torch.randn(B, T, N, C, generator=g).double()
    Wu, Wv = torch.randn(C, hg, generator=g).double() * 0.4, torch.randn(C, hg, generator=g).double() * 0.4
    P = PS.generator(X, Wu, Wv, 3.0, rowptr, col)
    assert P.shape == (B, col.numel())
    for b in range(B):
        torch.testing.assert_close(P[b], M.sparse_generator(X[b:b + 1], Wu, Wv, 3.0, rowptr, col), rtol=1e-12,
                                   atol=1e-14)
    # the windows do not see each other: the batch-summed generator differs from every per-window one
    Pb = M.sparse_generator(X, Wu, Wv, 3.0, rowptr, col)
    assert all(float((Pb - P[b]).abs().max()) > 1e-6 for b in range(B))
