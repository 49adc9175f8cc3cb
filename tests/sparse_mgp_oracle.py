"""The graph generator on a fixed CSR pattern, restated in fp64 on the CPU -- test infrastructure, like oracle/.

The dense generator (`stc_gnn_b200.mgp.pair_scores`, pinned to the reference's MGP_Gen in tests/test_multi_cpu.py) is
M - M^T followed by a row softmax of its relu.  Here the same score is evaluated at the stored edges of a pattern only
and each row is normalised over its stored edges; with a complete pattern the two are the same thing.  The edge
gathers below form [nnz, width] slabs: fine at test sizes, and exactly what the CUDA path avoids."""
import torch

Tensor = torch.Tensor


def edge_rows(rowptr: Tensor) -> Tensor:
    return torch.repeat_interleave(torch.arange(rowptr.numel() - 1), (rowptr[1:] - rowptr[:-1]).long())


def node_major(X_seq: Tensor, W: Tensor, alpha: float) -> Tensor:
    """tanh(alpha X W) as [N, B*T*hg] (node-major), X_seq [B, T, N, C]."""
    B, T, N, C = X_seq.shape
    return torch.tanh(alpha * (X_seq @ W)).permute(2, 0, 1, 3).reshape(N, -1)


def pair_scores_at(U: Tensor, V: Tensor, rowptr: Tensor, col: Tensor) -> Tensor:
    """S[e] = <U_n, V_m> - <V_n, U_m> for every stored edge e = (n, m), CSR order."""
    n, m = edge_rows(rowptr), col.long()
    return (U[n] * V[m]).sum(-1) - (V[n] * U[m]).sum(-1)


def edge_softmax(S: Tensor, rowptr: Tensor) -> Tensor:
    """Softmax of relu(S) over the stored edges of each row (the max is subtracted, as torch.softmax does)."""
    N = rowptr.numel() - 1
    rows = edge_rows(rowptr)
    r = torch.relu(S)
    mx = torch.zeros(N, dtype=S.dtype).scatter_reduce(0, rows, r.detach(), "amax", include_self=True)
    ex = torch.exp(r - mx[rows])
    den = torch.zeros(N, dtype=S.dtype).index_add(0, rows, ex)
    return ex / den[rows]


def sparse_generator(X_seq: Tensor, Wu: Tensor, Wv: Tensor, alpha: float, rowptr: Tensor, col: Tensor) -> Tensor:
    """P [nnz]: the generated edge values of the pattern (rowptr, col)."""
    return edge_softmax(pair_scores_at(node_major(X_seq, Wu, alpha), node_major(X_seq, Wv, alpha), rowptr, col), rowptr)


def complete_pattern(N: int):
    rowptr = torch.arange(N + 1, dtype=torch.int32) * N
    return rowptr, torch.arange(N, dtype=torch.int32).repeat(N)


def random_pattern(N: int, deg: int, seed: int, empty_every: int = 0, hub=None, self_loop_every: int = 3):
    """CSR (rowptr, col) int32: distinct sorted neighbours per row drawn at random (so the pattern is asymmetric), rows
    without edges (every `empty_every`-th), a self-loop in every `self_loop_every`-th non-empty row, optionally one row
    `hub[0]` linked to `hub[1]` nodes."""
    g = torch.Generator().manual_seed(seed)
    rows = []
    for n in range(N):
        d = hub[1] if hub is not None and n == hub[0] else int(torch.randint(1, deg + 1, (1,), generator=g))
        if empty_every and n % empty_every == 1:
            rows.append(torch.zeros(0, dtype=torch.long))
            continue
        nb = torch.randperm(N, generator=g)[:d]
        nb = nb[nb != n]
        if self_loop_every and n % self_loop_every == 0:
            nb = torch.cat([nb, torch.tensor([n])])
        rows.append(torch.sort(nb).values)
    col = torch.cat(rows).to(torch.int32)
    rowptr = torch.zeros(N + 1, dtype=torch.int32)
    rowptr[1:] = torch.cumsum(torch.tensor([r.numel() for r in rows]), 0)
    return rowptr, col


def drop_near_zero_scores(rowptr: Tensor, col: Tensor, S: Tensor, rel: float = 1e-3):
    """The pattern without the edges (other than self-loops) whose score is within rel * mean|S| of 0: there a relu
    boundary flip between fp32 and fp64 would decide the comparison.  Returns (rowptr, col, number dropped)."""
    rows = edge_rows(rowptr)
    keep = (S.abs() >= rel * S.abs().mean()) | (rows == col.long())
    counts = torch.bincount(rows[keep], minlength=rowptr.numel() - 1)
    new_rowptr = torch.zeros_like(rowptr)
    new_rowptr[1:] = torch.cumsum(counts, 0).to(rowptr.dtype)
    return new_rowptr, col[keep].contiguous(), int((~keep).sum())


def dense_of(rowptr: Tensor, col: Tensor, vals: Tensor, N: int) -> Tensor:
    G = torch.zeros(N, N, dtype=vals.dtype)
    return G.index_put((edge_rows(rowptr), col.long()), vals, accumulate=True)
