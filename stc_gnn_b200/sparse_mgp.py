"""The reference's spatial graph generator on a fixed sparsity pattern (the large-N form of `MGP_Gen`).

`MGP_Gen` (STC_GNN.py:210-243) builds a dense [N, N] support from the input window every forward:
`U = tanh(alpha X Wu)`, `V = tanh(alpha X Wv)`, `M[i,j] = sum_{b,t,h} U[b,t,i,h] V[b,t,j,h]`,
`Ps = softmax(relu(M - M^T), dim=-1)`.  On a graph of 65,536 nodes that matrix cannot exist.  Here the same pair score
is evaluated only at the stored edges of a fixed pattern (a kNN or grid adjacency), and each row is normalised over
its stored edges:

    S[e] = M[n,m] - M[m,n] = <U_n, V_m> - <V_n, U_m>      every stored edge e = (n, m), Gs-CSR order
    P[e] = exp(relu(S[e])) / sum_{e' in row n} exp(relu(S[e']))

and the result is the pattern carrying P: a learnable `CsrSupport` whose edge gradient, returned by the cell, flows
back into `Wu`, `Wv`.  On a pattern that stores all N^2 entries this is exactly the reference's `Ps`.  Entries off the
pattern are excluded from the softmax, not counted as exp(0) as the dense softmax counts them.  There is no sparse
counterpart of `MixedFusion`: mixing a prior's values with P is the caller's choice, made on [nnz] tensors.

The scores and the softmax are CUDA kernels (stc_pair_scores_csr, stc_edge_softmax_fwd / _bwd) that read each node's
U / V row and keep only [nnz] vectors; nothing of size [nnz, width] is formed.  The gradient of the scores is four plain
CSR hops: with D = the pattern carrying dS, dU = (D - D^T) V and dV = (D^T - D) U.
"""
from __future__ import annotations

import torch
from torch import nn

from . import _lib, mgp
from .support import CsrSupport, support_apply


def _check_pattern(pattern, N: int, who: str) -> None:
    if not isinstance(pattern, CsrSupport):
        raise RuntimeError(f"{who}: the pattern must be a CsrSupport, got {type(pattern).__name__}")
    if pattern.N != N:
        raise RuntimeError(f"{who}: the pattern has {pattern.N} nodes, the input {N}")


class _PairScores(torch.autograd.Function):
    """S[e] = <U_n, V_m> - <V_n, U_m> at the pattern's stored edges; U, V [N, width]."""

    @staticmethod
    def forward(ctx, U, V, pattern):
        lib = _lib.load()
        N, width = U.shape
        S = torch.empty(pattern.nnz, dtype=torch.float32, device=U.device)
        _lib.check(lib.stc_pair_scores_csr(pattern.struct(), N, width, U.data_ptr(), V.data_ptr(), S.data_ptr(),
                                           torch.cuda.current_stream().cuda_stream), "stc_pair_scores_csr")
        ctx.save_for_backward(U, V)
        ctx.pattern = pattern
        return S

    @staticmethod
    def backward(ctx, dS):
        U, V = ctx.saved_tensors
        D = ctx.pattern.with_values(dS.detach())

        def skew(A, sign):   # sign * (D - D^T) A, as [N, width]
            Y = support_apply(D, A[None], transpose=False, alpha=sign)
            return support_apply(D, A[None], transpose=True, alpha=-sign, beta=1.0, Z=Y, out=Y)[0]

        dU = skew(V, 1.0) if ctx.needs_input_grad[0] else None
        dV = skew(U, -1.0) if ctx.needs_input_grad[1] else None
        return dU, dV, None


class _EdgeSoftmax(torch.autograd.Function):
    """P = softmax of relu(S) over each row's stored edges."""

    @staticmethod
    def forward(ctx, S, pattern):
        lib = _lib.load()
        P = torch.empty_like(S)
        _lib.check(lib.stc_edge_softmax_fwd(pattern.struct(), pattern.N, S.data_ptr(), P.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream), "stc_edge_softmax_fwd")
        ctx.save_for_backward(S, P)
        ctx.pattern = pattern
        return P

    @staticmethod
    def backward(ctx, dP):
        S, P = ctx.saved_tensors
        dPc = dP.contiguous()
        dS = torch.empty_like(S)
        _lib.check(_lib.load().stc_edge_softmax_bwd(ctx.pattern.struct(), ctx.pattern.N, S.data_ptr(), P.data_ptr(),
                                                    dPc.data_ptr(), dS.data_ptr(),
                                                    torch.cuda.current_stream().cuda_stream), "stc_edge_softmax_bwd")
        return dS, None


def pair_softmax_csr(U: torch.Tensor, V: torch.Tensor, pattern: CsrSupport, group=None, average: bool = False):
    """P [nnz] (Gs-CSR order of `pattern`): the row softmax over stored edges of relu(<U_n,V_m> - <V_n,U_m>).

    U, V: [N, width] float32 CUDA tensors (node-major; width = B*T*hg for the generator).  Only the pattern's
    structure is used; its values are never read.  Differentiable w.r.t. U and V.

    With a process group (batch data-parallel: each rank holds a shard of the batch, so its U, V are the shard's
    columns) the partial scores are summed over the ranks before the softmax (`mgp.sum_forward`) and the gradient
    arriving at P is all-reduced (`mgp.reduce_grad`), as `mgp.mgp_forward_dp` does for the dense generator: every rank
    gets the global-batch P, and the gradients of what produced U, V are this shard's partial sums for the caller's
    `dp.GradBucket` (`average`: the bucket is averaged).  [nnz] floats are communicated each way."""
    for name, t in (("U", U), ("V", V)):
        if not t.is_cuda or t.dtype != torch.float32 or t.dim() != 2:
            raise RuntimeError(f"pair_softmax_csr: {name} must be a [N, width] float32 CUDA tensor (there is no CPU "
                               f"path), got {tuple(t.shape)} {t.dtype} on {t.device}")
    if U.shape != V.shape or U.device != V.device:
        raise RuntimeError(f"pair_softmax_csr: U {tuple(U.shape)} on {U.device} and V {tuple(V.shape)} on {V.device} "
                           f"must match")
    _check_pattern(pattern, U.shape[0], "pair_softmax_csr")
    if pattern.device != U.device:
        raise RuntimeError(f"pair_softmax_csr: the pattern lives on {pattern.device}, U on {U.device}")
    S = _PairScores.apply(U.contiguous(), V.contiguous(), pattern)
    S = mgp.sum_forward(S, group, average)
    return mgp.reduce_grad(_EdgeSoftmax.apply(S, pattern), group, average)


class SparseGraphGenerator(nn.Module):
    """The spatial half of the reference's `MGP_Gen` on a fixed CSR pattern: forward(X_seq, pattern) returns the
    pattern carrying the generated edge values, a `CsrSupport` the cell learns through.

    `params_S` has the reference's names, shapes and initialisation (`Wu`, `Wv`: [num_categories, hidden_dim],
    xavier-normal), so a reference checkpoint's `mix_graph_pair.params_S.*` entries load with strict=True once the
    `mix_graph_pair.` prefix is stripped.  The parameters do not depend on N: a generator trained on one graph loads
    onto another with the same number of categories."""

    def __init__(self, num_categories: int, hidden_dim: int, alpha: float = 3):
        super().__init__()
        self.alpha = alpha
        self.params_S = nn.ParameterDict({"Wu": nn.Parameter(torch.randn(num_categories, hidden_dim)),
                                          "Wv": nn.Parameter(torch.randn(num_categories, hidden_dim))})
        for p in self.params_S.values():
            nn.init.xavier_normal_(p)

    def forward(self, X_seq: torch.Tensor, pattern: CsrSupport, group=None, average: bool = False) -> CsrSupport:
        """X_seq [B, T, N, C] float32 CUDA -> `pattern.with_values(P)`.  Under torch.no_grad() the values do not require
        grad and the cell treats the support as constant.  `group` / `average`: batch data-parallel, as in
        `pair_softmax_csr` (X_seq is this rank's shard)."""
        Wu, Wv = self.params_S["Wu"], self.params_S["Wv"]
        if not X_seq.is_cuda or X_seq.dtype != torch.float32 or X_seq.dim() != 4:
            raise RuntimeError(f"SparseGraphGenerator: X_seq must be a [B, T, N, C] float32 CUDA tensor (there is no "
                               f"CPU path), got {tuple(X_seq.shape)} {X_seq.dtype} on {X_seq.device}")
        B, T, N, C = X_seq.shape
        _check_pattern(pattern, N, "SparseGraphGenerator")
        if C != Wu.shape[0]:
            raise RuntimeError(f"SparseGraphGenerator: X_seq has {C} categories, params_S.Wu expects {Wu.shape[0]}")
        if X_seq.device != Wu.device or pattern.device != Wu.device:
            raise RuntimeError(f"SparseGraphGenerator: X_seq ({X_seq.device}), the pattern ({pattern.device}) and the "
                               f"parameters ({Wu.device}) must share a device")
        Xn = X_seq.permute(2, 0, 1, 3).reshape(N, B * T, C)       # node-major copy of the small input
        U = torch.tanh(self.alpha * (Xn @ Wu)).reshape(N, -1)      # [N, B*T*hg], contiguous
        V = torch.tanh(self.alpha * (Xn @ Wv)).reshape(N, -1)
        return pattern.with_values(pair_softmax_csr(U, V, pattern, group, average))
