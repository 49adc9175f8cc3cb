"""Learnable edge values on a row-partitioned CSR support, CPU side (no GPU needed):

* the value maps of `halo.PartitionedSupport` (adjoint slices, forward gather map) on patterns with explicit zeros,
  empty rows and an asymmetric pattern, at world 1-4;
* the edge gradient of `halo.adjoint_chain_ext` through those maps, over `gloo` at world 2 and 3, against fp64
  autograd of the unpartitioned spatial recurrence.

The arithmetic here is fp64 torch (an injected hop); the product arithmetic is CUDA-only.
"""
import pytest
import torch
import torch.distributed as dist

from oracle import stc_oracle as O
from stc_gnn_b200 import halo
from tests.test_multi_cpu import run_ranks


def pattern(N, seed, deg=5, empty_every=6, zero_frac=0.2):
    """CSR (rowptr, col, vals) of a structurally asymmetric pattern: distinct sorted neighbours per row, every
    `empty_every`-th row empty, about `zero_frac` of the edges stored as 0, a few edges across every block boundary."""
    g = torch.Generator().manual_seed(seed)
    rows = []
    for n in range(N):
        d = 0 if n % empty_every == 2 else int(torch.randint(1, deg + 1, (1,), generator=g))
        nb = torch.randperm(N, generator=g)[:d]
        if d:
            nb = torch.cat([nb, torch.tensor([(n + 1) % N])])
        rows.append(torch.unique(nb))
    col = torch.cat(rows)
    rowptr = torch.zeros(N + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(torch.tensor([r.numel() for r in rows]), 0)
    vals = torch.rand(col.numel(), generator=g, dtype=torch.float64) + 0.25
    vals[torch.rand(col.numel(), generator=g) < zero_frac] = 0.0
    return rowptr, col, vals


def edge_rows(rowptr):
    return torch.repeat_interleave(torch.arange(rowptr.numel() - 1), rowptr[1:] - rowptr[:-1])


def dense_of(rowptr, col, vals, N):
    """Dense Gs[n, m] from CSR, differentiable w.r.t. vals."""
    G = torch.zeros(N, N, dtype=vals.dtype)
    return G.index_put((edge_rows(rowptr), col), vals, accumulate=True)


def local_dense(rowptr, col, vals, nrows, ncols):
    G = torch.zeros(nrows, ncols, dtype=vals.dtype)
    return G.index_put((edge_rows(rowptr[:nrows + 1]), col), vals, accumulate=True)


def learnable_partition(rowptr, col, vals, N, rank, world, group=None):
    return halo.PartitionedSupport(rowptr, col, vals.clone().requires_grad_(True), N, rank, world, group)


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("N,seed", [(37, 1), (50, 2)])
def test_value_maps_rebuild_the_local_operators(world, N, seed):
    rowptr, col, vals = pattern(N, seed)
    assert (vals == 0).any() and (rowptr[1:] == rowptr[:-1]).any()
    G0 = dense_of(rowptr, col, vals, N)
    assert not torch.equal(G0 != 0, (G0 != 0).t())
    nnz = col.numel()
    parts = [learnable_partition(rowptr, col, vals, N, r, world) for r in range(world)]
    assert all(p.learnable and p.fwd.op_val is None for p in parts)
    maps = [p.maps() for p in parts]
    # the adjoint slices partition [0, nnz) in rank order
    assert maps[0].edge_lo == 0 and maps[-1].edge_hi == nnz
    assert all(a.edge_hi == b.edge_lo for a, b in zip(maps, maps[1:]))
    # the forward maps, concatenated over the ranks, are the Gs^T order of the unpartitioned CsrSupport (t_perm)
    t_perm = torch.sort(col * N + edge_rows(rowptr), stable=True).indices
    assert torch.equal(torch.cat([m.fwd_ids for m in maps]), t_perm)
    v = torch.randn(nnz, generator=torch.Generator().manual_seed(seed + 100), dtype=torch.float64)
    G = dense_of(rowptr, col, v, N)
    for p, m in zip(parts, maps):
        ext = torch.cat([torch.arange(p.start, p.start + p.nloc), p.fwd.halo_global])
        nx = p.fwd.next
        assert m.bwd_rowptr.numel() == nx + 1 and m.fwd_rowptr.numel() == nx + 1
        assert int(m.bwd_rowptr[p.nloc]) == int(m.bwd_rowptr[-1]) == m.edge_hi - m.edge_lo   # halo rows: no edges
        assert int(m.fwd_rowptr[p.nloc]) == int(m.fwd_rowptr[-1]) == m.fwd_ids.numel()
        bwd = local_dense(m.bwd_rowptr, m.bwd_col, v[m.edge_lo:m.edge_hi], p.nloc, nx)
        fwd = local_dense(m.fwd_rowptr, m.fwd_col, v[m.fwd_ids], p.nloc, nx)
        rows = slice(p.start, p.start + p.nloc)
        torch.testing.assert_close(bwd, G[rows][:, ext], rtol=0, atol=0)
        torch.testing.assert_close(fwd, G.t()[rows][:, ext], rtol=0, atol=0)
        # every forward row lists its edges by ascending global source node
        n_glob = ext[m.fwd_col]
        for r in range(p.nloc):
            seg = n_glob[m.fwd_rowptr[r]:m.fwd_rowptr[r + 1]]
            assert bool((seg[1:] >= seg[:-1]).all())


def test_with_values_keeps_plans_and_maps():
    rowptr, col, vals = pattern(30, 3)
    const = halo.PartitionedSupport(rowptr, col, vals, 30, 0, 2)
    assert not const.learnable and const.fwd.op_val is not None
    v = torch.rand(col.numel(), dtype=torch.float64, requires_grad=True)
    ps = const.with_values(torch.nn.functional.softplus(v))
    assert ps.learnable and not const.learnable and ps.fwd is const.fwd and ps.maps() is const.maps()
    with pytest.raises(RuntimeError, match="nnz"):
        const.with_values(v[:-1])
    with pytest.raises(RuntimeError, match="nnz"):
        halo.PartitionedSupport(rowptr, col, v[1:], 30, 0, 2)


def _learned_hop(ps, v):
    """CPU stand-in for PartitionedSupport.hop_ext on a learnable support: the real in-place halo refresh, the local
    operators rebuilt from the values `v` through the maps, the edge gradient formed per stored edge."""
    m = ps.maps()

    def hop(X_ext, out_ext, Z_ext, alpha, beta, direction, *, A_ext=None, coef=1.0, dvals=None):
        plan = ps.fwd if direction == "fwd" else ps.bwd
        B = X_ext.shape[0]
        X3 = X_ext.view(B, plan.next, -1)
        halo.exchange_into(plan, X3, ps.group)
        rp, c, val = ((m.fwd_rowptr, m.fwd_col, v[m.fwd_ids]) if direction == "fwd"
                      else (m.bwd_rowptr, m.bwd_col, v[m.edge_lo:m.edge_hi]))
        A = local_dense(rp, c, val, plan.nloc, plan.next)
        Y = alpha * torch.einsum("nm,bmw->bnw", A, X3)
        if beta != 0.0:
            Y = Y + beta * Z_ext.view(B, plan.next, -1)[:, :plan.nloc]
        if dvals is not None:
            r = edge_rows(rp[:plan.nloc + 1])
            A3 = A_ext.reshape(B, plan.next, -1)
            dvals += coef * (A3[:, r] * X3[:, c]).sum(dim=(0, 2))
        out_ext.view(B, plan.next, -1)[:, :plan.nloc] = Y
    return hop


def _edge_grad_chain_case(rank, world):
    """adjoint_chain_ext with terms + dvals, summed over the ranks == autograd of the unpartitioned recurrence."""
    N, B, C, L, Ks = 41, 2, 3, 2, 4
    rowptr, col, vals = pattern(N, seed=7)
    v = vals.clone().requires_grad_(True)
    g = torch.Generator().manual_seed(8)
    X = torch.randn(B, N, C, L, generator=g, dtype=torch.float64)
    dY = [torch.randn(B, N, C, L, generator=g, dtype=torch.float64) for _ in range(Ks)]
    terms = O.spatial_terms(X, dense_of(rowptr, col, v, N), Ks)
    sum((t * d).sum() for t, d in zip(terms, dY)).backward()
    ps = learnable_partition(rowptr, col, vals, N, rank, world)
    assert ps.fwd.nhalo > 0
    hop = _learned_hop(ps, vals)
    ne, lo = ps.fwd.next, ps.start
    junk = lambda: torch.full((B, ne, C, L), 7.0, dtype=torch.float64)   # halo rows the chain must never read
    # forward terms through the same in-place hop (the values through the forward map)
    ext = [junk() for _ in range(Ks)]
    ext[0][:, :ps.nloc] = ps.local_slice(X)
    for k in range(1, Ks):
        hop(ext[k - 1], ext[k], None if k == 1 else ext[k - 2], 1.0 if k == 1 else 2.0, 0.0 if k == 1 else -1.0, "fwd")
        O.assert_close(ext[k][:, :ps.nloc], ps.local_slice(terms[k].detach()), f"forward term {k} (rank {rank})",
                       1e-9, 1e-10)
    ybar = []
    for d in dY:
        e = junk()
        e[:, :ps.nloc] = ps.local_slice(d)
        ybar.append(e)
    m = ps.maps()
    dvals = torch.zeros(col.numel(), dtype=torch.float64)
    got = halo.adjoint_chain_ext(ps, ybar, hop=hop, terms=ext[:Ks - 1], dvals=dvals[m.edge_lo:m.edge_hi])
    assert not dvals[:m.edge_lo].any() and not dvals[m.edge_hi:].any(), "a rank writes its own slice only"
    dist.all_reduce(dvals)
    torch.testing.assert_close(dvals, v.grad, rtol=1e-9, atol=1e-9 * float(v.grad.abs().max()))
    assert float(dvals[vals == 0].abs().min()) > 0.0, "an edge stored as 0 still gets a gradient"
    # the chain without an edge gradient (the positional hop signature) is unchanged
    Xg = X.clone().requires_grad_(True)
    sum((t * d).sum() for t, d in zip(O.spatial_terms(Xg, dense_of(rowptr, col, vals, N), Ks), dY)).backward()
    O.assert_close(got[:, :ps.nloc], ps.local_slice(Xg.grad), f"adjoint chain (rank {rank}, lo {lo})", 1e-9, 1e-10)


@pytest.mark.parametrize("world", [2, 3])
def test_partitioned_edge_gradient_chain_matches_autograd(world):
    run_ranks(_edge_grad_chain_case, world)
