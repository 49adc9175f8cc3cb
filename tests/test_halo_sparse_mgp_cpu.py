"""The generator on a row-partitioned pattern, CPU side (no GPU needed): the padded all-gather layout of [nnz] edge
vectors (`halo.ValueMaps.edge_bounds / edge_pad`, `halo.gather_edges`) at world 1-4 on patterns with empty rows, a
rank whose rows store no edges, self-loops and asymmetry, and over gloo at world 2 and 3: the gathered vector and the
backward of the gather (this rank's slice of the incoming gradient, nothing communicated).

The scores, the softmax and their adjoint are CUDA-only; tests/test_halo_sparse_mgp_gpu.py checks them."""
import pytest
import torch

from stc_gnn_b200 import halo
from stc_gnn_b200.dp import shard_bounds
from tests import sparse_mgp_oracle as SO
from tests.test_multi_cpu import run_ranks

N = 31


def pattern(seed, empty_block_of=None):
    """Asymmetric CSR (rowptr, col): every 4th row empty, self-loops; `empty_block_of = (rank, world)`: that rank's
    rows store no edges at all."""
    rowptr, col = SO.random_pattern(N, 5, seed=seed, empty_every=4)
    rowptr, col = rowptr.long(), col.long()
    if empty_block_of is not None:
        s, e = shard_bounds(N, *empty_block_of)
        keep = ~((SO.edge_rows(rowptr) >= s) & (SO.edge_rows(rowptr) < e))
        counts = torch.bincount(SO.edge_rows(rowptr)[keep], minlength=N)
        rowptr = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(counts, 0)])
        col = col[keep]
    return rowptr, col


def partition(rowptr, col, rank, world, group=None):
    vals = torch.rand(col.numel(), dtype=torch.float64).requires_grad_(True)
    return halo.PartitionedSupport(rowptr, col, vals, N, rank, world, group)


CASES = [(1, None), (2, (1, 3)), (3, (1, 3))]


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("seed,empty", CASES)
def test_padded_gather_layout_reproduces_the_vector(world, seed, empty):
    rowptr, col = pattern(seed, empty)
    nnz = col.numel()
    G = SO.dense_of(rowptr, col, torch.ones(nnz, dtype=torch.float64), N)
    assert not torch.equal(G != 0, (G != 0).t()) and (rowptr[1:] == rowptr[:-1]).any()
    assert bool((SO.edge_rows(rowptr) == col).any()), "self-loops"
    parts = [partition(rowptr, col, r, world) for r in range(world)]
    maps = [p.maps() for p in parts]
    if empty is not None and world == 3:
        assert maps[1].edge_lo == maps[1].edge_hi, "rank 1 stores no edges"
    for m in maps:
        assert m.edge_bounds == [(mm.edge_lo, mm.edge_hi) for mm in maps]
        assert m.edge_pad == max(hi - lo for lo, hi in m.edge_bounds)
    x = torch.randn(nnz, dtype=torch.float64, generator=torch.Generator().manual_seed(seed))
    # what the all-gather produces: every rank's slice, zero-padded to edge_pad, in rank order
    buf = torch.cat([torch.cat([x[m.edge_lo:m.edge_hi], x.new_zeros(m.edge_pad - (m.edge_hi - m.edge_lo))])
                     for m in maps])
    assert buf.numel() == world * maps[0].edge_pad
    for p, m in zip(parts, maps):
        assert torch.equal(halo.unpad_edges(p, buf), x)
        assert torch.equal(buf[m.padded_index(torch.arange(nnz))], x)
        assert torch.equal(buf[m.padded_index(m.fwd_ids)], x[m.fwd_ids]), "forward operator values, padded"
    # the halo of the asymmetric pattern is symmetric: it holds nodes the rank's rows do not read themselves (the
    # in-neighbours the transpose term of the backward reads)
    if world > 1:
        reads = lambda p, m: set(m.bwd_col[m.bwd_col >= p.nloc].tolist())
        assert any(len(reads(p, m)) < p.fwd.nhalo for p, m in zip(parts, maps))


def _gather_case(rank, world):
    for seed, empty in CASES:
        rowptr, col = pattern(seed, empty)
        nnz = col.numel()
        ps = partition(rowptr, col, rank, world)
        m = ps.maps()
        x = torch.randn(nnz, dtype=torch.float64, generator=torch.Generator().manual_seed(seed))
        x_loc = x[m.edge_lo:m.edge_hi].clone().requires_grad_(True)
        full = halo.gather_edges(ps, x_loc)
        assert torch.equal(full, x), f"gathered vector (rank {rank}/{world}, seed {seed})"
        g = torch.randn(nnz, dtype=torch.float64, generator=torch.Generator().manual_seed(100 + rank))
        full.backward(g)               # a different gradient on every rank: only the own slice may come back
        assert torch.equal(x_loc.grad, g[m.edge_lo:m.edge_hi]), f"gather backward (rank {rank}/{world})"
        out, work = halo.gather_edges_padded(ps, x_loc.detach())
        assert work is None and out.numel() == world * m.edge_pad
        pad = out.view(world, m.edge_pad)
        for r, (lo, hi) in enumerate(m.edge_bounds):
            assert not pad[r, hi - lo:].any(), "padding is zeros"


@pytest.mark.parametrize("world", [2, 3])
def test_gather_edges_over_gloo(world):
    run_ranks(_gather_case, world)


def test_gather_edges_world_one_is_the_identity():
    rowptr, col = pattern(1)
    ps = partition(rowptr, col, 0, 1)
    x = torch.randn(col.numel(), dtype=torch.float64)
    assert halo.gather_edges(ps, x) is x
