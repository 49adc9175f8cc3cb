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

On a row-partitioned graph (`halo.PartitionedSupport`) each rank holds its node block of X_seq.  A row's scores and
softmax read only that row's node and its out-neighbours, so [U | V] of the halo nodes is exchanged once, through the
same overlap skeleton as a partitioned hop (stc_pair_scores_csr_rows scores the interior rows meanwhile), and each
rank's slice P[edge_lo:edge_hi] is all-gathered into the full [nnz] P.  The backward needs no reduction of dP (the
gradient arriving at P is exact on the rank's rows) and one all-gather of dS for the transpose term
(`pair_softmax_partitioned`).  At world 1 it is bitwise the unpartitioned generator.

The pattern may also be chosen from the scores themselves (`gen(X_seq, k=k)`, `topk_pattern`): with
S[n, m] = <U_n, V_m> - <V_n, U_m> for EVERY m (m = n included, whose score is exactly 0),

    selection  row n stores the k columns with the largest S[n, m]; equal scores go to the smaller column; columns are
               stored in ascending order, every row has exactly k edges (1 <= k <= min(N, 32)), rowptr = k * arange(N+1)
    values     exactly those of the fixed-pattern generator on the selected pattern: stc_pair_scores_csr recomputes the
               scores in fp32 and stc_edge_softmax_fwd takes the softmax of their relu over the k stored edges, so
               gen(X_seq, k=k) is bitwise gen(X_seq, pattern=<the selected pattern>), and with k = N it is the
               reference's dense Ps
    gradient   flows through the values only: the selection is piecewise constant in U, V and gets no gradient, as in
               any top-k graph learner

The selection is the CUDA kernel stc_pair_topk: all N^2 scores as 128 x 128 tiles of one 3xTF32 tensor-core GEMM
[U | V] [V | -U]^T, each row's k best kept on chip, so memory stays O(N k) where the score matrix alone would take
4 N^2 bytes (17 GB at N = 65,536).  Its output is a pure function of (U, V, k): bitwise the same on every call.  A
score within the 3xTF32 rounding (about 1e-6 relative) of a row's k-th score may be ranked differently from an fp64
evaluation.

The selection also runs on the row-partitioned graph (`gen(X_seq_block, k=k, partition=halo.RowPartition(N, rank,
world))`): every rank all-gathers U, V of all N nodes (detached; [N, width] each), selects its own rows over all N
columns (`pair_topk(..., rows=(start, nloc))`, stc_pair_topk_rows: each row bitwise that row of the full selection),
all-gathers the [N, k] selection and partitions it on the device (`RowPartition.support`, one small device-to-host
copy), then forms P exactly as on a fixed partitioned pattern.  Scores of unrelated nodes pick neighbours anywhere in
the graph, so the halo of a selected pattern can approach every remote node: each hop then moves close to an
all-gather.
"""
from __future__ import annotations

import torch
from torch import nn

from . import _lib, halo, mgp
from .halo import PartitionedSupport
from .support import CsrSupport, support_apply

TOPK_MAX = 32   # stc_pair_topk keeps at most this many columns a row on chip


def _check_pattern(pattern, N: int, who: str) -> None:
    if isinstance(pattern, PartitionedSupport):
        if pattern.nloc != N:
            raise RuntimeError(f"{who}: this rank's block of the pattern has {pattern.nloc} nodes, the input {N}")
        return
    if not isinstance(pattern, CsrSupport):
        raise RuntimeError(f"{who}: the pattern must be a CsrSupport or a halo.PartitionedSupport, got "
                           f"{type(pattern).__name__}")
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


def pair_scores_rows(pattern: CsrSupport, width: int, ld: int, U: torch.Tensor, V: torch.Tensor, scores: torch.Tensor,
                     rows: torch.Tensor) -> None:
    """stc_pair_scores_csr_rows: scores[e] for the edges of the listed rows of `pattern` only (the other entries of
    `scores` are left as they are).  U, V: views whose row n starts at data_ptr + n * ld floats (e.g. the two halves
    of one [N, 2 * width] buffer); rows: int32 CUDA tensor."""
    if rows.dtype != torch.int32 or not rows.is_cuda or not rows.is_contiguous():
        raise RuntimeError("pair_scores_rows: `rows` must be a contiguous int32 CUDA tensor")
    if rows.numel() == 0 or pattern.nnz == 0:
        return
    _lib.check(_lib.load().stc_pair_scores_csr_rows(pattern.struct(), pattern.N, width, ld, U.data_ptr(), V.data_ptr(),
                                                    scores.data_ptr(), rows.data_ptr(), rows.numel(),
                                                    torch.cuda.current_stream().cuda_stream), "stc_pair_scores_csr_rows")


class _PartitionedPairSoftmax(torch.autograd.Function):
    """P[edge_lo:edge_hi] (this rank's slice, Gs-CSR order) from this rank's U, V [nloc, width]; see
    `pair_softmax_partitioned`."""

    @staticmethod
    def forward(ctx, U, V, ps):
        lib = _lib.load()
        n, W = U.shape
        ne = ps.fwd.next
        m = ps.maps()
        stream = torch.cuda.current_stream().cuda_stream
        UV = U.new_empty(ne, 2 * W)              # [U | V] of [local | halo] nodes: one exchange moves both
        UV[:n, :W] = U
        UV[:n, W:] = V
        Sc = U.new_empty(m.edge_hi - m.edge_lo)
        op = ps.local_operator("bwd", Sc)        # rows: this rank's nodes, edges in Gs-CSR order (pattern only)
        every = None
        if ps.world == 1:                        # the skeleton's launch(None): every row
            every = ps._dev.get(("rows", str(U.device)))
            if every is None:
                every = ps._dev[("rows", str(U.device))] = torch.arange(ne, dtype=torch.int32, device=U.device)
        Vv = UV[:, W:]
        # the halo rows are refreshed on the adjoint plan (the operator Gs: row n reads its out-neighbours m); the halo
        # is symmetric, so they also hold the in-neighbours the backward's transpose term reads
        ps._overlapped("bwd", UV.view(1, ne, 2 * W),
                       lambda rows: pair_scores_rows(op, W, 2 * W, UV, Vv, Sc, every if rows is None else rows))
        P = torch.empty_like(Sc)
        if Sc.numel():
            _lib.check(lib.stc_edge_softmax_fwd(op.struct(), ne, Sc.data_ptr(), P.data_ptr(), stream),
                       "stc_edge_softmax_fwd")
        ctx.save_for_backward(UV, Sc, P)
        ctx.ps = ps
        return P

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dP):
        UV, Sc, P = ctx.saved_tensors
        ps = ctx.ps
        m = ps.maps()
        ne, W2 = UV.shape
        W, n = W2 // 2, ps.nloc
        dS = torch.empty_like(Sc)
        if Sc.numel():
            dPc = dP.contiguous()
            _lib.check(_lib.load().stc_edge_softmax_bwd(ps.local_operator("bwd", dS).struct(), ne, Sc.data_ptr(),
                                                        P.data_ptr(), dPc.data_ptr(), dS.data_ptr(),
                                                        torch.cuda.current_stream().cuda_stream),
                       "stc_edge_softmax_bwd")
        # with D = the pattern carrying dS: [dU | dV] = (D - D^T) [V | -U].  This rank's rows of D are the adjoint local
        # operator carrying dS (own edges); its rows of D^T are the forward local operator, whose edges other ranks own:
        # dS of every edge is all-gathered while D [U | V] runs.  Both read only the halo rows the forward refreshed.
        if ps.world > 1:
            buf, work = halo.gather_edges_padded(ps, dS, async_op=True)
        X = UV.view(1, ne, W2)
        Z = torch.zeros_like(X) if dS.numel() == 0 else support_apply(ps.local_operator("bwd", dS), X, transpose=False)
        fwd_ids = ps._operator_structure("fwd", UV.device)[2]
        if ps.world > 1:
            work.wait()
            key = ("padded_fwd_ids", str(UV.device))
            idx = ps._dev.get(key)
            if idx is None:
                idx = ps._dev[key] = m.padded_index(m.fwd_ids).to(UV.device)
            dS_fwd = buf[idx]
        else:
            dS_fwd = dS[fwd_ids]
        if dS_fwd.numel():
            support_apply(ps.local_operator("fwd", dS_fwd), X, transpose=False, alpha=-1.0, beta=1.0, Z=Z, out=Z)
        Z = Z[0, :n]                             # [D U - D^T U | D V - D^T V] = [-dV | dU]
        return Z[:, W:].contiguous(), -Z[:, :W].contiguous(), None


def pair_softmax_partitioned(U_loc: torch.Tensor, V_loc: torch.Tensor, ps: PartitionedSupport) -> torch.Tensor:
    """`pair_softmax_csr` on a row-partitioned pattern: P [nnz], the full vector in Gs-CSR order, the same bytes on
    every rank.  U_loc, V_loc: [nloc, width] float32 CUDA, this rank's nodes (`ps.local_slice`).  Every rank must call
    it, and run the backward, because both contain collectives (none at world 1).

    A row's scores and softmax read that row's node and its out-neighbours: [U | V] of the halo nodes is exchanged once,
    on the adjoint plan of `ps`, and the rows whose neighbours are all local are scored while it is in flight
    (stc_pair_scores_csr_rows over the adjoint local operator, then stc_edge_softmax_fwd).  The rank's slice
    P[edge_lo:edge_hi] is all-gathered ([nnz] floats).  Backward: the gradient of the slice is the slice of the gradient
    arriving at P, with no communication (`halo.gather_edges` states what that requires of the caller); dS of every
    edge is all-gathered once for the transpose term of dU, dV.  The gradients of U_loc, V_loc are exact and local."""
    for name, t in (("U", U_loc), ("V", V_loc)):
        if not t.is_cuda or t.dtype != torch.float32 or t.dim() != 2:
            raise RuntimeError(f"pair_softmax_partitioned: {name} must be a [nloc, width] float32 CUDA tensor (there is "
                               f"no CPU path), got {tuple(t.shape)} {t.dtype} on {t.device}")
    if U_loc.shape != V_loc.shape or U_loc.device != V_loc.device:
        raise RuntimeError(f"pair_softmax_partitioned: U {tuple(U_loc.shape)} on {U_loc.device} and V "
                           f"{tuple(V_loc.shape)} on {V_loc.device} must match")
    _check_pattern(ps, U_loc.shape[0], "pair_softmax_partitioned")
    P_loc = _PartitionedPairSoftmax.apply(U_loc.contiguous(), V_loc.contiguous(), ps)
    return halo.gather_edges(ps, P_loc)


def _check_topk_args(N: int, k, who: str) -> None:
    if isinstance(k, bool) or not isinstance(k, int):
        raise RuntimeError(f"{who}: k must be an int, got {type(k).__name__}")
    if k < 1 or k > TOPK_MAX or k > N:
        raise RuntimeError(f"{who}: k = {k} outside [1, min(N = {N}, {TOPK_MAX})]")


def pair_topk(U: torch.Tensor, V: torch.Tensor, k: int, scores: bool = False, rows=None):
    """cols [N, k] int32: the k columns m of each row n with the largest S[n, m] = <U_n, V_m> - <V_n, U_m> over all N
    candidates (S[n, n] = 0; ties to the smaller column), ascending in each row (stc_pair_topk).  With `scores`, also
    the matching S values [N, k] (float32, 3xTF32).  U, V: [N, width] float32 CUDA; a width that is not a multiple of 4
    is padded with zero columns, which add nothing to any score.  A NaN score (NaN or inf in U / V) ranks, and is
    reported, as -inf, so every row still gets k distinct columns in [0, N).  Not differentiable: the result is an
    index set.

    `rows=(row0, n_rows)`: only the rows [row0, row0 + n_rows), still scored against all N columns
    (stc_pair_topk_rows); the result is [n_rows, k] and bitwise those rows of the full selection."""
    for name, t in (("U", U), ("V", V)):
        if t.dtype != torch.float32 or t.dim() != 2:
            raise RuntimeError(f"pair_topk: {name} must be a [N, width] float32 CUDA tensor, got {tuple(t.shape)} "
                               f"{t.dtype}")
    if U.shape != V.shape or U.device != V.device:
        raise RuntimeError(f"pair_topk: U {tuple(U.shape)} on {U.device} and V {tuple(V.shape)} on {V.device} must match")
    N, width = U.shape
    _check_topk_args(N, k, "pair_topk")
    row0, n_rows = (0, N) if rows is None else (int(rows[0]), int(rows[1]))
    if row0 < 0 or n_rows < 0 or row0 + n_rows > N:
        raise RuntimeError(f"pair_topk: rows [{row0}, {row0} + {n_rows}) outside [0, N = {N})")
    if not U.is_cuda:
        raise RuntimeError(f"pair_topk: U, V live on {U.device} (there is no CPU path)")
    if width == 0:
        raise RuntimeError("pair_topk: width must be positive")
    pad = -width % 4
    U, V = (torch.nn.functional.pad(t.detach(), (0, pad)) if pad else t.detach().contiguous() for t in (U, V))
    U, V = (t if t.data_ptr() % 16 == 0 else t.clone() for t in (U, V))
    lib = _lib.load()
    cols = torch.empty(n_rows, k, dtype=torch.int32, device=U.device)
    sc = torch.empty(n_rows, k, dtype=torch.float32, device=U.device) if scores else None
    stream = torch.cuda.current_stream().cuda_stream
    if rows is None:
        ws_bytes = lib.stc_pair_topk_workspace_bytes(N, width + pad, k)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=U.device)
        _lib.check(lib.stc_pair_topk(N, width + pad, U.data_ptr(), V.data_ptr(), k, cols.data_ptr(),
                                     sc.data_ptr() if scores else None, ws.data_ptr(), ws_bytes, stream), "stc_pair_topk")
    elif n_rows:
        ws_bytes = lib.stc_pair_topk_rows_workspace_bytes(N, width + pad, n_rows, k)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=U.device)
        _lib.check(lib.stc_pair_topk_rows(N, width + pad, U.data_ptr(), V.data_ptr(), row0, n_rows, k, cols.data_ptr(),
                                          sc.data_ptr() if scores else None, ws.data_ptr(), ws_bytes, stream),
                   "stc_pair_topk_rows")
    return (cols, sc) if scores else cols


def topk_pattern(U: torch.Tensor, V: torch.Tensor, k: int) -> CsrSupport:
    """The k-regular pattern `pair_topk` selects, as a `CsrSupport` with zero values and its Gs^T permutation, built on
    the device with no host synchronisation."""
    return CsrSupport._k_regular(pair_topk(U, V, k))


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

    def forward(self, X_seq: torch.Tensor, pattern=None, group=None, average: bool = False, k: int = None,
                partition: halo.RowPartition = None):
        """X_seq [B, T, N, C] float32 CUDA -> `pattern.with_values(P)`.  Under torch.no_grad() the values do not require
        grad and the cell treats the support as constant.  `group` / `average`: batch data-parallel, as in
        `pair_softmax_csr` (X_seq is this rank's shard).

        `pattern` may also be a `halo.PartitionedSupport` (the graph's rows split over the ranks): X_seq is then this
        rank's node block [B, T, nloc, C] (the batch is replicated), P is formed by `pair_softmax_partitioned` and the
        result is the partitioned pattern carrying the full P.  Every rank runs the forward and the backward.  Wu, Wv
        are replicated and their gradients are partial sums over the rank's nodes: with `pattern.reduce_per_cell`
        (default) the backward all-reduces them, so `.grad` is the full gradient on every rank; without it the partial
        sums are left for the caller's `dp.GradBucket`, as for the cell.  The gradient of X_seq is exact, with no
        communication.  Batch data-parallelism (`group`, `average`) cannot be combined with the row partition.

        `k` instead of `pattern`: the pattern is chosen from the scores, the k largest of every row over all N columns
        (`topk_pattern` on U, V detached; module docstring), and P is formed on it as on a fixed pattern.  The result is
        a k-regular `CsrSupport`.  Not combinable with batch data-parallelism, nor with a fixed `PartitionedSupport`.

        `k` with `partition` (a `halo.RowPartition`): the same selection on the row-partitioned graph.  X_seq is this
        rank's node block [B, T, nloc, C]; U, V of every node are all-gathered (detached), the rank selects its own rows
        (`pair_topk(..., rows=(start, nloc))`), the [N, k] selection is all-gathered and partitioned on the device
        (`partition.support`), and P is formed on it exactly as on a fixed partitioned pattern (gradients, the Wu / Wv
        reduction by `partition.reduce_per_cell`, the no-grad path).  The result is a `PartitionedSupport`; every rank
        runs the forward and the backward."""
        Wu, Wv = self.params_S["Wu"], self.params_S["Wv"]
        partitioned = isinstance(pattern, PartitionedSupport)
        if partition is not None:
            if not isinstance(partition, halo.RowPartition):
                raise RuntimeError(f"SparseGraphGenerator: partition must be a halo.RowPartition, got "
                                   f"{type(partition).__name__}")
            if k is None or pattern is not None:
                raise RuntimeError("SparseGraphGenerator: partition= selects the pattern on the row-partitioned graph: "
                                   "give k=, and no pattern")
            if group is not None or average:
                raise RuntimeError("SparseGraphGenerator: batch data-parallelism (group= / average=) cannot be combined "
                                   "with a row partition")
        if k is not None:
            if partitioned:
                raise RuntimeError("SparseGraphGenerator: k= selects the pattern on one device; a row-partitioned "
                                   "pattern cannot be combined with it")
            if group is not None or average:
                raise RuntimeError("SparseGraphGenerator: k= cannot be combined with batch data-parallelism "
                                   "(group= / average=): every rank would select from its own shard's scores")
        both = "SparseGraphGenerator: give exactly one of `pattern` (a fixed pattern) and `k` (select the k best " \
               "columns of every row)"
        if pattern is not None and k is not None:
            raise RuntimeError(both)
        if partitioned and (group is not None or average):
            raise RuntimeError("SparseGraphGenerator: batch data-parallelism (group= / average=) cannot be combined "
                               "with a row-partitioned pattern")
        if not X_seq.is_cuda or X_seq.dtype != torch.float32 or X_seq.dim() != 4:
            raise RuntimeError(f"SparseGraphGenerator: X_seq must be a [B, T, N, C] float32 CUDA tensor (there is no "
                               f"CPU path), got {tuple(X_seq.shape)} {X_seq.dtype} on {X_seq.device}")
        if pattern is None and k is None:
            raise RuntimeError(both)
        B, T, N, C = X_seq.shape
        if partition is not None:
            if N != partition.nloc:
                raise RuntimeError(f"SparseGraphGenerator: this rank's block of the partition has {partition.nloc} "
                                   f"nodes, the input {N}")
            _check_topk_args(partition.N, k, "SparseGraphGenerator")
        elif k is not None:
            _check_topk_args(N, k, "SparseGraphGenerator")
        else:
            _check_pattern(pattern, N, "SparseGraphGenerator")
        if C != Wu.shape[0]:
            raise RuntimeError(f"SparseGraphGenerator: X_seq has {C} categories, params_S.Wu expects {Wu.shape[0]}")
        if X_seq.device != Wu.device or (pattern is not None and not partitioned and pattern.device != Wu.device):
            where = "" if pattern is None else f", the pattern ({pattern.device})"
            raise RuntimeError(f"SparseGraphGenerator: X_seq ({X_seq.device}){where} and the parameters ({Wu.device}) "
                               f"must share a device")
        rows_split = pattern if partitioned else partition
        if rows_split is not None and rows_split.reduce_per_cell and rows_split.world > 1:
            Wu, Wv = mgp.reduce_grad(Wu, rows_split.group), mgp.reduce_grad(Wv, rows_split.group)
        Xn = X_seq.permute(2, 0, 1, 3).reshape(N, B * T, C)       # node-major copy of the small input
        U = torch.tanh(self.alpha * (Xn @ Wu)).reshape(N, -1)      # [N, B*T*hg], contiguous
        V = torch.tanh(self.alpha * (Xn @ Wv)).reshape(N, -1)
        if partition is not None:
            W = U.shape[1]
            UV = partition.gather_rows(torch.cat([U.detach(), V.detach()], 1))   # [N, 2W]: every node's U, V
            sel = pair_topk(UV[:, :W], UV[:, W:], k, rows=(partition.start, partition.nloc))
            pattern = partition.support(partition.gather_rows(sel))
            partitioned = True
        if partitioned:
            return pattern.with_values(pair_softmax_partitioned(U, V, pattern))
        if k is not None:
            pattern = topk_pattern(U.detach(), V.detach(), k)
        return pattern.with_values(pair_softmax_csr(U, V, pattern, group, average))
