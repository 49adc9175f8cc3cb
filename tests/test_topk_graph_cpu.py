"""The sparse generator's pattern selection without a GPU: the fp64 selection oracle (tests/topk_graph_oracle.py), the
k-regular structure `topk_pattern` builds against what `CsrSupport` builds from the same (rowptr, col), and the
generator's argument errors that are raised before anything touches a device."""
import pytest
import torch

from oracle import stc_oracle as O
from stc_gnn_b200 import mgp
from stc_gnn_b200.halo import PartitionedSupport
from stc_gnn_b200.sparse_mgp import SparseGraphGenerator, pair_topk
from stc_gnn_b200.support import CsrSupport, k_regular_structure
from tests import sparse_mgp_oracle as SO
from tests import topk_graph_oracle as TO


def test_selection_ranks_and_breaks_ties_by_column():
    S = torch.tensor([[0.0, 3.0, 1.0, 3.0, -2.0, 1.0],
                      [5.0, 0.0, 5.0, 5.0, 5.0, -1.0],
                      [-1.0, -1.0, 0.0, -3.0, -1.0, -2.0]], dtype=torch.float64)
    assert TO.select(S, 1).tolist() == [[1], [0], [2]]
    assert TO.select(S, 2).tolist() == [[1, 3], [0, 2], [0, 2]]
    assert TO.select(S, 3).tolist() == [[1, 2, 3], [0, 2, 3], [0, 1, 2]]
    assert TO.check_selection(S, TO.select(S, 3), 3) == 3      # every row ties at its 3rd score
    with pytest.raises(AssertionError, match="row 0"):
        TO.check_selection(S, torch.tensor([[1, 3, 4], [0, 2, 3], [0, 1, 2]]), 3)


def test_scores_are_antisymmetric_with_an_exact_zero_diagonal():
    g = torch.Generator().manual_seed(1)
    U, V = torch.randn(30, 7, generator=g, dtype=torch.float64), torch.randn(30, 7, generator=g, dtype=torch.float64)
    S = TO.full_scores(U, V)
    assert torch.all(S.diagonal() == 0)
    torch.testing.assert_close(S, -S.t(), rtol=0, atol=1e-12)
    torch.testing.assert_close(TO.full_scores(U, V, torch.tensor([4, 9])), S[[4, 9]], rtol=0, atol=1e-12)
    # the diagonal competes like any other score
    U2 = torch.zeros(3, 1, dtype=torch.float64)
    assert TO.select(TO.full_scores(U2, U2), 1).tolist() == [[0], [0], [0]]   # every score 0: the smallest column


def test_k_equal_n_is_the_complete_pattern_and_the_dense_generator():
    B, T, N, C, hg, alpha = 2, 3, 17, 4, 5, 3.0
    g = torch.Generator().manual_seed(5)
    X = torch.randn(B, T, N, C, generator=g, dtype=torch.float64)
    Wu = torch.randn(C, hg, generator=g, dtype=torch.float64) * 0.3
    Wv = torch.randn(C, hg, generator=g, dtype=torch.float64) * 0.3
    U, V = SO.node_major(X, Wu, alpha), SO.node_major(X, Wv, alpha)
    cols = TO.select(TO.full_scores(U, V), N)
    rowptr, col = SO.complete_pattern(N)
    assert torch.equal(cols.reshape(-1).int(), col)
    P = SO.sparse_generator(X, Wu, Wv, alpha, rowptr, col).reshape(N, N)
    Ps = torch.softmax(torch.relu(mgp.pair_scores(X, Wu, Wv, alpha)), -1)
    O.assert_close(P, Ps, "k = N vs the dense generator", rtol=1e-12, atol_scale=1e-12)


@pytest.mark.parametrize("N,k", [(1, 1), (9, 3), (40, 7), (64, 32)])
def test_k_regular_structure_matches_csr_support(N, k):
    g = torch.Generator().manual_seed(N + k)
    cols = torch.sort(torch.stack([torch.randperm(N, generator=g)[:k] for _ in range(N)]), dim=1).values.int()
    rowptr, col, t_rowptr, t_col, t_perm = k_regular_structure(cols)
    assert torch.equal(rowptr, (torch.arange(N + 1) * k).int()) and torch.equal(col, cols.reshape(-1))
    ref = CsrSupport.__new__(CsrSupport)         # the learnable constructor's transpose, run on the host
    ref.N, ref.rowptr, ref.col, ref.device, ref._t_struct = N, rowptr, col, torch.device("cpu"), None
    want = ref._transpose_structure()
    for name, a, b in zip(("t_rowptr", "t_col", "t_perm"), (t_rowptr, t_col, t_perm), want):
        assert a.dtype == b.dtype and torch.equal(a, b), name
    dense = torch.zeros(N, N)
    dense[torch.arange(N).repeat_interleave(k), col.long()] = torch.arange(N * k, dtype=torch.float32) + 1
    vals = (torch.arange(N * k, dtype=torch.float32) + 1)[t_perm]           # Gs^T-CSR values through the permutation
    t_rows = torch.repeat_interleave(torch.arange(N), (t_rowptr[1:] - t_rowptr[:-1]).long())
    assert torch.equal(dense.t()[t_rows, t_col.long()], vals)


def test_generator_argument_errors_before_any_device_work():
    gen = SparseGraphGenerator(4, 8)
    X = torch.randn(2, 3, 20, 4)
    with pytest.raises(RuntimeError, match="exactly one of `pattern`"):
        gen(X, CsrSupport.__new__(CsrSupport), k=4)
    with pytest.raises(RuntimeError, match="row-partitioned"):
        gen(X, PartitionedSupport.__new__(PartitionedSupport), k=4)
    with pytest.raises(RuntimeError, match="batch data-parallelism"):
        gen(X, k=4, group=object())
    with pytest.raises(RuntimeError, match="batch data-parallelism"):
        gen(X, k=4, average=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        gen(X, k=4)
    U = torch.zeros(20, 6)
    for bad in (0, 33, 21):
        with pytest.raises(RuntimeError, match=f"k = {bad} outside"):
            pair_topk(U, U, bad)
    with pytest.raises(RuntimeError, match="no CPU path"):
        pair_topk(U, U, 4)
    with pytest.raises(RuntimeError, match="float32"):
        pair_topk(U.double(), U.double(), 4)
