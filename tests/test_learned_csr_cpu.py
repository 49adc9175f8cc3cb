"""Learnable edge values of a CSR spatial support, CPU side: the analytic edge-value gradient (the gradient the fused
adjoint hop accumulates, tests/learned_csr_oracle.py) against fp64 autograd of the dense oracle, sampled at the
pattern."""
import pytest
import torch

from tests.helpers import oracle_cell_with_grads, random_case
from tests.learned_csr_oracle import edge_pattern, stc_cell_edge_grad


def pattern_with_zero_edges(N, deg, seed):
    """CSR (rowptr, col, vals) with `deg` distinct neighbours per row (some rows with none) and about one edge in
    five stored with the value 0.  Built from rowptr / col, since a dense-to-sparse conversion would drop those."""
    g = torch.Generator().manual_seed(seed)
    rows = []
    for n in range(N):
        d = 0 if n % 7 == 3 else int(torch.randint(1, deg + 1, (1,), generator=g))
        rows.append(torch.sort(torch.randperm(N, generator=g)[:d]).values)
    col = torch.cat(rows)
    rowptr = torch.zeros(N + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(torch.tensor([r.numel() for r in rows]), 0)
    vals = (torch.rand(col.numel(), generator=g) + 0.5) / deg
    vals[torch.rand(col.numel(), generator=g) < 0.2] = 0.0
    return rowptr, col, vals.double()


@pytest.mark.parametrize("Ks", [1, 2, 3, 4])
@pytest.mark.parametrize("Kc", [1, 2, 3])
def test_oracle_edge_gradient_is_dense_dGs_at_the_pattern(Ks, Kc):
    B, N, C, Din, h = 2, 23, 3, 2, 4
    rowptr, col, vals = pattern_with_zero_edges(N, 4, seed=10 * Ks + Kc)
    assert (vals == 0).any() and (rowptr[1:] == rowptr[:-1]).any()
    Gs = torch.sparse_csr_tensor(rowptr, col, vals, size=(N, N))
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=Ks * 3 + Kc)
    t["Gs"] = Gs
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, activation=None)
    _, g_ref = oracle_cell_with_grads(t, cfg)       # fp64 autograd through the DENSE Gs
    dv = stc_cell_edge_grad(Gs, t["Gc"], t["Xt"], t["H"], t["Wg"], t["bg"], t["Wc"], t["bc"], Ks, Kc, t["dHn"])
    row, c = edge_pattern(Gs)
    assert torch.equal(c, col)
    want = g_ref["dGs"][row, c]
    if Ks == 1:   # no spatial hop: the support does not enter the cell
        assert float(dv.abs().max()) == 0.0 and float(want.abs().max()) == 0.0
        return
    torch.testing.assert_close(dv, want, rtol=1e-10, atol=1e-12)
    assert float(dv[vals == 0].abs().min()) > 0.0, "an edge stored as 0 still gets a gradient"


def test_edge_pattern_of_coo_and_csr_agree():
    rowptr, col, vals = pattern_with_zero_edges(15, 4, seed=4)
    G = torch.sparse_csr_tensor(rowptr, col, vals, size=(15, 15))
    r1, c1 = edge_pattern(G)
    r2, c2 = edge_pattern(G.to_sparse_coo())
    assert torch.equal(r1, r2) and torch.equal(c1, c2) and r1.numel() == vals.numel()
