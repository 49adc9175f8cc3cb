"""The fp64 restatement of the generator on a fixed CSR pattern (tests/sparse_mgp_oracle.py) against the dense
generator `mgp.pair_scores` (pinned to the reference's MGP_Gen in tests/test_multi_cpu.py), and the module's surface.
No GPU needed."""
import inspect

import pytest
import torch

import stc_gnn_b200 as S
from stc_gnn_b200 import mgp
from tests import sparse_mgp_oracle as SO
from tests.helpers import import_reference

ALPHA = 3.0


def _inputs(B, T, N, C, hg, seed):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(B, T, N, C, generator=g, dtype=torch.float64)
    Wu = torch.randn(C, hg, generator=g, dtype=torch.float64) * 0.3
    Wv = torch.randn(C, hg, generator=g, dtype=torch.float64) * 0.3
    return X, Wu, Wv


def test_complete_pattern_is_the_dense_generator():
    B, T, N, C, hg = 3, 4, 17, 5, 6
    X, Wu, Wv = _inputs(B, T, N, C, hg, seed=1)
    rowptr, col = SO.complete_pattern(N)
    got = SO.sparse_generator(X, Wu, Wv, ALPHA, rowptr, col).reshape(N, N)
    want = torch.softmax(torch.relu(mgp.pair_scores(X, Wu, Wv, ALPHA)), -1)
    assert (got - want).abs().max().item() < 1e-12
    assert torch.all(torch.diagonal(SO.pair_scores_at(SO.node_major(X, Wu, ALPHA), SO.node_major(X, Wv, ALPHA),
                                                      rowptr, col).reshape(N, N)) == 0.0)


def test_complete_pattern_gradients_are_the_dense_generators():
    B, T, N, C, hg = 2, 3, 11, 4, 5
    X, Wu0, Wv0 = _inputs(B, T, N, C, hg, seed=2)
    w = torch.randn(N, N, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    rowptr, col = SO.complete_pattern(N)
    grads = []
    for fn in (lambda Wu, Wv: SO.sparse_generator(X, Wu, Wv, ALPHA, rowptr, col).reshape(N, N),
               lambda Wu, Wv: torch.softmax(torch.relu(mgp.pair_scores(X, Wu, Wv, ALPHA)), -1)):
        Wu, Wv = Wu0.clone().requires_grad_(True), Wv0.clone().requires_grad_(True)
        (fn(Wu, Wv) * w).sum().backward()
        grads.append((Wu.grad, Wv.grad))
    for a, b in zip(grads[0], grads[1]):
        assert (a - b).abs().max().item() < 1e-12 * max(1.0, b.abs().max().item())


def test_partial_pattern_is_the_dense_score_normalised_over_stored_edges():
    """Empty rows, self-loops, an asymmetric pattern and a hub row: P[e] = exp(relu(Sd[n,m])) / sum over row n's stored
    edges of the same, with Sd the dense M - M^T; a self-loop scores exactly 0; an empty row gets nothing; the values a
    pattern stores (explicit zeros included) play no part, since only (rowptr, col) is an input."""
    B, T, N, C, hg = 2, 5, 40, 3, 4
    X, Wu, Wv = _inputs(B, T, N, C, hg, seed=4)
    rowptr, col = SO.random_pattern(N, 6, seed=5, empty_every=7, hub=(9, 35))
    rows = SO.edge_rows(rowptr)
    A = torch.zeros(N, N, dtype=torch.bool)
    A[rows, col.long()] = True
    assert not torch.equal(A, A.t()), "the pattern must be asymmetric"
    assert (rowptr[1:] == rowptr[:-1]).any(), "the pattern must have empty rows"
    U, V = SO.node_major(X, Wu, ALPHA), SO.node_major(X, Wv, ALPHA)
    Sd = mgp.pair_scores(X, Wu, Wv, ALPHA)
    Se = SO.pair_scores_at(U, V, rowptr, col)
    assert (Se - Sd[rows, col.long()]).abs().max().item() < 1e-12
    loops = rows == col.long()
    assert loops.sum() > 0 and torch.all(Se[loops] == 0.0)
    P = SO.edge_softmax(Se, rowptr)
    ex = torch.where(A, torch.exp(torch.relu(Sd)), torch.zeros_like(Sd))
    want = (ex / ex.sum(-1, keepdim=True).clamp_min(1e-300))[rows, col.long()]
    assert (P - want).abs().max().item() < 1e-12
    rowsum = torch.zeros(N, dtype=torch.float64).index_add(0, rows, P)
    nonempty = rowptr[1:] > rowptr[:-1]
    assert torch.allclose(rowsum[nonempty], torch.ones(int(nonempty.sum()), dtype=torch.float64))
    assert torch.all(rowsum[~nonempty] == 0.0) and P.numel() == col.numel()


def test_dropping_near_zero_scores_keeps_self_loops():
    X, Wu, Wv = _inputs(2, 3, 30, 3, 4, seed=6)
    rowptr, col = SO.random_pattern(30, 8, seed=7, self_loop_every=1)
    S_ = SO.pair_scores_at(SO.node_major(X, Wu, ALPHA), SO.node_major(X, Wv, ALPHA), rowptr, col)
    r2, c2, dropped = SO.drop_near_zero_scores(rowptr, col, S_, rel=0.2)
    assert dropped > 0 and int(r2[-1]) == c2.numel() == col.numel() - dropped
    S2 = SO.pair_scores_at(SO.node_major(X, Wu, ALPHA), SO.node_major(X, Wv, ALPHA), r2, c2)
    loops = SO.edge_rows(r2) == c2.long()
    assert int(loops.sum()) == 30 and torch.all(S2[~loops].abs() >= 0.2 * S_.abs().mean())


def test_generator_surface():
    gen = S.SparseGraphGenerator(5, 16)
    sd = gen.state_dict()
    assert list(sd.keys()) == ["params_S.Wu", "params_S.Wv"]
    assert all(tuple(v.shape) == (5, 16) for v in sd.values())
    assert gen.alpha == inspect.signature(S.SparseGraphGenerator).parameters["alpha"].default
    with pytest.raises(RuntimeError, match="no CPU path"):
        gen(torch.zeros(2, 3, 4, 5), pattern=None)
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.pair_softmax_csr(torch.zeros(4, 6), torch.zeros(4, 6), None)


def test_generator_parameters_match_the_reference():
    """Names, shapes, initialisation and the alpha default of the reference's MGP_Gen.params_S: a reference
    checkpoint's `mix_graph_pair.params_S.*` entries load with strict=True."""
    ref, _ = import_reference()
    if ref is None:
        pytest.skip("needs the live reference")
    assert inspect.signature(ref.MGP_Gen).parameters["alpha"].default == \
        inspect.signature(S.SparseGraphGenerator).parameters["alpha"].default
    torch.manual_seed(11)
    rg = ref.MGP_Gen(num_nodes=12, num_categories=4, hidden_dim=6)
    torch.manual_seed(11)
    ours = S.SparseGraphGenerator(4, 6)
    want = {k: v for k, v in rg.state_dict().items() if k.startswith("params_S.")}
    assert list(want) == list(ours.state_dict())
    for k, v in want.items():
        assert torch.equal(v, ours.state_dict()[k]), k
    ours.load_state_dict(want, strict=True)
