"""The partition of a selected (k-regular) pattern, CPU side (no GPU needed): `PartitionedSupport.k_regular` on CPU
tensors against the host constructor on the same pattern, field for field (both plans, `maps()`, the exchange state),
for N in {1, 7, 61, 300}, k in {1, 4, 8}, world 1-4 (N < world leaves ranks without nodes) and every rank, on random
selections and on a selection that reads no remote column; `RowPartition.gather_rows` over gloo; the C-ABI prototypes
of the row-block selection.

The selection itself and the generator on the row partition are CUDA-only; tests/test_topk_halo_gpu.py checks them."""
import os
import re

import pytest
import torch

from stc_gnn_b200 import _lib, halo
from stc_gnn_b200.dp import shard_bounds
from tests.test_multi_cpu import run_ranks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def random_selection(N, k, seed):
    """[N, k] int32, k distinct columns a row, ascending (what `pair_topk` returns)."""
    g = torch.Generator().manual_seed(seed)
    return torch.sort(torch.rand(N, N, generator=g).argsort(1)[:, :k], 1).values.to(torch.int32)


def local_selection(N, k, world):
    """Every row selects columns of its own block only (nothing remote); a block smaller than k repeats no column, so
    such rows take the block and then the nearest columns of the next ones -- rows of blocks with >= k nodes stay
    local."""
    cols = torch.empty(N, k, dtype=torch.int64)
    for r in range(world):
        s, e = shard_bounds(N, r, world)
        for n in range(s, e):
            pool = list(range(s, e)) + [c for c in range(N) if c < s or c >= e]
            cols[n] = torch.tensor(sorted(pool[:k]))
    return cols.to(torch.int32)


def host_partition(cols, rank, world):
    N, k = cols.shape
    return halo.PartitionedSupport(torch.arange(N + 1) * k, cols.reshape(-1).long(), torch.zeros(N * k), N, rank,
                                   world)


def assert_same(a, b, what):
    assert isinstance(b, torch.Tensor), what
    assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b), f"{what}: {a} != {b}"


def assert_same_partition(got, want, tag):
    for name in ("N", "rank", "world", "nnz", "start", "nloc", "reduce_per_cell"):
        assert getattr(got, name) == getattr(want, name), (tag, name)
    assert got.vals is None and want.vals is None
    assert_same(got._rowptr, want._rowptr, f"rowptr {tag}")
    assert_same(got._col, want._col, f"col {tag}")
    for d in ("fwd", "bwd"):
        pg, pw = getattr(got, d), getattr(want, d)
        for name in ("rank", "world", "start", "nloc", "nhalo", "recv_counts", "send_counts", "next"):
            assert getattr(pg, name) == getattr(pw, name), (tag, d, name, getattr(pg, name), getattr(pw, name))
        assert len(pg.send_idx) == len(pw.send_idx) == pw.world
        for p, (a, b) in enumerate(zip(pg.send_idx, pw.send_idx)):
            assert_same(a, b, f"{d} send_idx[{p}] {tag}")
        for name in ("halo_global", "op_row", "op_col", "op_val"):
            assert_same(getattr(pg, name), getattr(pw, name), f"{d} {name} {tag}")
        sg, sw = got._device_state(d, "cpu"), want._device_state(d, "cpu")
        assert sg["nsend"] == sw["nsend"], tag
        for name in ("send_idx", "interior", "boundary"):
            assert_same(sg[name], sw[name], f"{d} exchange {name} {tag}")
    mg, mw = got.maps(), want.maps()
    for name in ("edge_lo", "edge_hi", "edge_bounds", "edge_pad"):
        assert getattr(mg, name) == getattr(mw, name), (tag, name)
    for name in ("bwd_rowptr", "bwd_col", "fwd_rowptr", "fwd_col", "fwd_ids"):
        assert_same(getattr(mg, name), getattr(mw, name), f"maps {name} {tag}")
    ids = torch.arange(want.nnz)
    assert_same(mg.padded_index(ids), mw.padded_index(ids), f"padded_index {tag}")


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("N,k", [(N, k) for N in (1, 7, 61, 300) for k in (1, 4, 8) if k <= N])
def test_k_regular_partition_is_the_host_partition(N, k, world):
    for kind, cols in (("random", random_selection(N, k, 100 * N + 10 * k + world)),
                       ("local", local_selection(N, k, world))):
        for rank in range(world):
            tag = f"({kind}, N {N}, k {k}, rank {rank}/{world})"
            got = halo.PartitionedSupport.k_regular(cols, rank, world)
            want = host_partition(cols, rank, world)
            assert_same_partition(got, want, tag)
            if kind == "local" and N >= world * k:
                assert got.fwd.nhalo == 0 and got.bwd.send_counts == [0] * world, tag


def test_row_partition_shares_its_state_and_reduce_flag():
    cols = random_selection(61, 4, 3)
    part = halo.RowPartition(61, 1, 3)
    part.reduce_per_cell = False
    a, b = part.support(cols), part.support(random_selection(61, 4, 4))
    assert (part.start, part.nloc) == (21, 20)
    assert not a.reduce_per_cell and a._streams is part._streams and b._streams is part._streams
    assert a.with_values(torch.zeros(61 * 4))._streams is part._streams
    with pytest.raises(RuntimeError, match="60 rows"):
        part.support(random_selection(60, 4, 3))


def _gather_rows_case(rank, world):
    for N in (7, 61, 47, 2):
        part = halo.RowPartition(N, rank, world)
        full = torch.arange(N * 3, dtype=torch.float64).view(N, 3) - 5.0
        got = part.gather_rows(full[part.start:part.start + part.nloc].clone())
        assert torch.equal(got, full), (N, rank, world)
        cols = full.to(torch.int32)
        assert torch.equal(part.gather_rows(cols[part.start:part.start + part.nloc].clone()), cols)


@pytest.mark.parametrize("world", [2, 3])
def test_gather_rows_over_gloo(world):
    run_ranks(_gather_rows_case, world)


def test_gather_rows_world_one_is_the_identity():
    x = torch.randn(5, 2)
    assert halo.RowPartition(5, 0, 1).gather_rows(x) is x


def _prototype_params(name):
    src = open(os.path.join(ROOT, "include", "stc_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^)]*)\)\s*;", src)
    assert m, name
    return [a.strip() for a in m.group(1).split(",")]


def test_abi_of_the_row_block_selection():
    lib = _lib.load()
    args = [a.split()[-1].lstrip("*") for a in _prototype_params("stc_pair_topk_rows")]
    assert args == ["N", "width", "u", "v", "row0", "n_rows", "k", "cols", "scores", "ws", "ws_bytes", "stream"]
    assert len(lib.stc_pair_topk_rows.argtypes) == len(args)
    ws = [a.split()[-1] for a in _prototype_params("stc_pair_topk_rows_workspace_bytes")]
    assert ws == ["N", "width", "n_rows", "k"] and len(lib.stc_pair_topk_rows_workspace_bytes.argtypes) == 4
    assert "stc_pair_topk_rows" in _lib.EXPORTED and "stc_pair_topk_rows_workspace_bytes" in _lib.EXPORTED
