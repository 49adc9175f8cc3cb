"""Per-sample spatial supports restated in fp64 on the CPU -- test infrastructure, like oracle/.

A per-sample CSR support carries values [B, nnz] on one pattern: sample b is hopped with its own Gs_b in every
Chebyshev term.  The cell is the oracle's own `stc_cell` with its spatial recurrence replaced by a batched one
(Y_1[b] = Gs_b^T X[b]), so autograd through it gives every gradient, the edge gradient [B, nnz] included.  The
generator restatement evaluates `tests/sparse_mgp_oracle.py` on each window's own U, V."""
import torch

from oracle import stc_oracle as O
from tests import sparse_mgp_oracle as M

Tensor = torch.Tensor


def dense_batch(rowptr: Tensor, col: Tensor, vals: Tensor, N: int) -> Tensor:
    """[B, N, N] with Gs_b[n, m] = vals[b, e] at the stored edges e = (n, m) (differentiable in vals)."""
    B = vals.shape[0]
    rows = M.edge_rows(rowptr)
    G = torch.zeros(B, N, N, dtype=vals.dtype)
    b = torch.arange(B)[:, None].expand(B, rows.numel())
    return G.index_put((b, rows[None].expand_as(b), col.long()[None].expand_as(b)), vals, accumulate=True)


def per_sample_terms(G: Tensor, Ks: int):
    """The spatial recurrence Y_k = 2 Gs_b^T Y_{k-1} - Y_{k-2} with one Gs_b per sample (G [B, N, N])."""
    def hop(X):
        return torch.einsum("bnm,bncl->bmcl", G, X)

    def terms(X):
        Y = [X]
        if Ks > 1:
            Y.append(hop(X))
        for _ in range(2, Ks):
            Y.append(2.0 * hop(Y[-1]) - Y[-2])
        return Y
    return terms


def cell_with_grads(t: dict, rowptr: Tensor, col: Tensor, vals: Tensor, Ks: int, Kc: int, activation=None):
    """(H', grads) of the per-sample cell in fp64 through autograd; grads has dvals [B, nnz] and the cell's others."""
    names = ["Gc", "Xt", "H", "Wg", "Wc"] + (["bg", "bc"] if t.get("bg") is not None else [])
    v = {k: t[k].double().clone().requires_grad_(True) for k in names}
    ev = vals.double().clone().requires_grad_(True)
    N = t["Xt"].shape[1]
    fn = per_sample_terms(dense_batch(rowptr, col, ev, N), Ks)
    Hn = O.stc_cell(None, v["Gc"], v["Xt"], v["H"], v["Wg"], v.get("bg"), v["Wc"], v.get("bc"), Ks, Kc, activation,
                    spatial_terms_fn=fn)
    Hn.backward(t["dHn"].double())
    z = lambda x: x.grad if x.grad is not None else torch.zeros_like(x)
    g = dict(dXt=z(v["Xt"]), dH=z(v["H"]), dWg=z(v["Wg"]), dWc=z(v["Wc"]), dGc=z(v["Gc"]), dvals=z(ev))
    if "bg" in v:
        g.update(dbg=z(v["bg"]), dbc=z(v["bc"]))
    return Hn.detach(), g


def generator(X_seq: Tensor, Wu: Tensor, Wv: Tensor, alpha: float, rowptr: Tensor, col: Tensor) -> Tensor:
    """P [B, nnz]: S_b[e = (n, m)] = sum_{t,h} U[b,t,n,h] V[b,t,m,h] - V[b,t,n,h] U[b,t,m,h] (no sum over the batch),
    then the softmax of relu(S_b) over row n's stored edges, for every sample at once."""
    U, V = torch.tanh(alpha * (X_seq @ Wu)), torch.tanh(alpha * (X_seq @ Wv))   # [B, T, N, hg]
    n, m = M.edge_rows(rowptr), col.long()
    S = torch.einsum("bteh,bteh->be", U[:, :, n], V[:, :, m]) - torch.einsum("bteh,bteh->be", V[:, :, n], U[:, :, m])
    return torch.stack([M.edge_softmax(s, rowptr) for s in S])
