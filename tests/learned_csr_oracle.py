"""Edge-value gradient of a sparse spatial support on the CPU (fp64) -- test infrastructure, like oracle/.

The analytic backward of oracle/stc_oracle.py (``stc_cell_backward``) walks the spatial recurrence in reverse and forms
dGs += coef * Y_{k-1} (x) ybar_k for a dense support only.  Here the same walk, built from the oracle's own pieces,
evaluates that product at the stored entries of a sparse Gs instead: the gradient w.r.t. its edge values, in CSR
order, which is what the fused adjoint hop (stc_support_apply_edge_grad) accumulates."""
from typing import Tuple

import torch

from oracle import stc_oracle as O

Tensor = torch.Tensor


def edge_pattern(G) -> Tuple[Tensor, Tensor]:
    """(row, col) of every stored entry of a torch sparse G, in CSR order (row-major; explicit zeros included)."""
    if G.layout == torch.sparse_csr:
        crow = G.crow_indices()
        row = torch.repeat_interleave(torch.arange(G.shape[0]), crow[1:] - crow[:-1])
        return row, G.col_indices()
    idx = G.to_sparse_coo().coalesce().indices()
    return idx[0], idx[1]


def bdg_dif_edge_grad(X: Tensor, Gs, Gc: Tensor, W: Tensor, dOut: Tensor, Ks: int, Kc: int) -> Tensor:
    """d(loss)/d(stored values of Gs) of the linear part of ``O.bdg_dif`` given dOut (pre-activation gradient)."""
    L, Hout = X.shape[-1], W.shape[1]
    Wv = W.reshape(Ks, Kc, L, Hout)
    Q = O.cheby_matrix_terms(Gc, Kc)
    Y = O.spatial_terms(X, Gs, Ks)
    ybar = []
    for n in range(Ks):
        dYn = torch.zeros_like(X)
        for c in range(Kc):
            dF = dOut @ Wv[n, c].t()
            dYn = dYn + (dF if c == 0 else torch.einsum("bmdl,cd->bmcl", dF, Q[c]))
        ybar.append(dYn)
    rows, cols = edge_pattern(Gs)
    # coef * sum_{b,c,l} Y[k-1][b,row,c,l] * ybar[k][b,col,c,l] at every stored edge (row, col)
    edge = lambda A, Bm: torch.einsum("becl,becl->e", A[:, rows], Bm[:, cols])
    dvals = torch.zeros(rows.numel(), dtype=X.dtype)
    for k in range(Ks - 1, 1, -1):
        dvals = dvals + 2.0 * edge(Y[k - 1], ybar[k])
        ybar[k - 1] = ybar[k - 1] + 2.0 * O.support_apply(Gs, ybar[k])
        ybar[k - 2] = ybar[k - 2] - ybar[k]
    if Ks > 1:
        dvals = dvals + edge(Y[0], ybar[1])
    return dvals


def stc_cell_edge_grad(Gs, Gc, Xt, H, Wg, bg, Wc, bc, Ks, Kc, dHn, activation=None) -> Tensor:
    """Gradient of ``O.stc_cell`` w.r.t. the stored edge values of a sparse Gs (CSR order), given dHn."""
    h, Din = H.shape[-1], Xt.shape[-1]
    _, u, r, c = O.stc_cell(Gs, Gc, Xt, H, Wg, bg, Wc, bc, Ks, Kc, activation, return_gates=True)
    du, dc = dHn * (c - H), dHn * u
    dpre_c = dc * (1.0 - c * c) * O._act_grad_mask(c, "tanh", activation)
    Xc = torch.cat([Xt, r * H], dim=-1)
    dv = bdg_dif_edge_grad(Xc, Gs, Gc, Wc, dpre_c, Ks, Kc)
    drH = O.bdg_dif_backward(Xc, Gs, Gc, Wc, dpre_c, Ks, Kc, need_dGs=False)[0][..., Din:]
    dr = drH * H
    dpre_g = torch.cat([du * u * (1.0 - u) * O._act_grad_mask(u, "sigmoid", activation),
                        dr * r * (1.0 - r) * O._act_grad_mask(r, "sigmoid", activation)], dim=-1)
    return dv + bdg_dif_edge_grad(torch.cat([Xt, H], dim=-1), Gs, Gc, Wg, dpre_g, Ks, Kc)
