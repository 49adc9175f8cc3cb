"""Spatial support handed to the cell: a dense [N,N] tensor (learned Gs, as MGP_Gen produces:
/root/reference/framework/STC_GNN.py:233) or a constant CSR graph (synthetic large-N configs)."""
from __future__ import annotations

import torch

from . import _lib


class CsrSupport:
    """Sparse spatial support Gs in CSR, together with Gs^T in CSR.

    The forward mode product contracts over Gs's first index (STC_GNN.py:37), so forward walks rows of
    Gs^T and backward walks rows of Gs; both are built once here.

    The sparsity pattern is fixed; the edge values may be learned.  When ``vals`` requires grad (an ``nn.Parameter``
    of shape [nnz], or a value computed from one, e.g. ``softplus(raw)``) the cell returns their gradient, in the order
    of ``vals`` (Gs-CSR order).  Every edge the pattern stores is trainable, including edges whose value is 0.
    ``t_perm`` maps Gs-CSR order to Gs^T-CSR order (``t_vals = vals[t_perm]``); the cell re-gathers ``t_vals`` before
    each forward, so an in-place update of ``vals`` is seen by the next step.  ``with_values(v)`` gives a support
    that shares the structure and the permutation with new values (values recomputed every step).
    """

    def __init__(self, rowptr: torch.Tensor, col: torch.Tensor, vals: torch.Tensor, num_nodes: int):
        if not (rowptr.is_cuda and col.is_cuda and vals.is_cuda):
            raise RuntimeError("CsrSupport tensors must live on a CUDA device (there is no CPU path)")
        self.N = int(num_nodes)
        self.rowptr = rowptr.to(torch.int32).contiguous()
        self.col = col.to(torch.int32).contiguous()
        self.vals = vals.to(torch.float32).contiguous()
        self.nnz = int(self.vals.numel())
        self.device = self.vals.device
        self.t_perm, self._t_struct = None, None
        if self.vals.requires_grad:
            if self.vals.dim() != 1 or self.nnz != self.col.numel() or self.nnz != int(self.rowptr[-1].item()):
                raise RuntimeError(f"CsrSupport: learnable values must be a [nnz] vector in the order of `col` "
                                   f"(nnz = {self.col.numel()}), got shape {tuple(self.vals.shape)}")
            self.t_rowptr, self.t_col, self.t_perm = self._transpose_structure()
            self.t_vals = torch.empty(self.nnz, dtype=torch.float32, device=self.device)
            self.sync_t_vals()
            return
        t = torch.sparse_csr_tensor(self.rowptr.long(), self.col.long(), self.vals, size=(self.N, self.N))
        tt = t.to_sparse_coo().t().coalesce().to_sparse_csr()
        self.t_rowptr = tt.crow_indices().to(torch.int32).contiguous()
        self.t_col = tt.col_indices().to(torch.int32).contiguous()
        self.t_vals = tt.values().to(torch.float32).contiguous()

    def _transpose_structure(self):
        """(t_rowptr, t_col, t_perm) of Gs^T from Gs's CSR, in integer arithmetic (computed once): Gs^T-CSR lists the
        edges sorted by (col, row), so t_perm is a stable argsort of col * N + row, and entry i of Gs^T is edge
        t_perm[i] of Gs.  Every stored edge is kept, whatever its value."""
        if self._t_struct is None:
            N, nnz = self.N, self.col.numel()
            row = torch.repeat_interleave(torch.arange(N, device=self.device, dtype=torch.int64),
                                          (self.rowptr[1:] - self.rowptr[:-1]).to(torch.int64), output_size=nnz)
            colL = self.col.to(torch.int64)
            t_perm = torch.sort(colL * N + row, stable=True).indices.contiguous()
            t_rowptr = torch.zeros(N + 1, dtype=torch.int64, device=self.device)
            t_rowptr[1:] = torch.cumsum(torch.bincount(colL, minlength=N), 0)
            self._t_struct = (t_rowptr.to(torch.int32).contiguous(), row[t_perm].to(torch.int32).contiguous(), t_perm)
        return self._t_struct

    @property
    def learnable(self) -> bool:
        """True when the edge values require grad (the cell then returns / accumulates their gradient)."""
        return self.vals.requires_grad

    def sync_t_vals(self) -> None:
        """t_vals = vals[t_perm] into the persistent Gs^T buffer, on the current stream (a CUDA-graph capture
        records the gather, so a replay sees the values as they are then)."""
        if self.t_perm is not None:
            torch.index_select(self.vals.detach(), 0, self.t_perm, out=self.t_vals)

    def with_values(self, vals: torch.Tensor) -> "CsrSupport":
        """A support with this one's pattern (and Gs^T permutation) and new edge values [nnz] (Gs-CSR order)."""
        v = vals.to(torch.float32).contiguous()
        if v.device != self.device or v.shape != (self.nnz,):
            raise RuntimeError(f"CsrSupport.with_values: values must be a [{self.nnz}] vector on {self.device}, got "
                               f"{tuple(v.shape)} on {v.device}")
        out = CsrSupport.__new__(CsrSupport)
        out.N, out.rowptr, out.col, out.vals, out.nnz, out.device = self.N, self.rowptr, self.col, v, self.nnz, self.device
        out._t_struct = self._transpose_structure()
        out.t_rowptr, out.t_col, out.t_perm = out._t_struct
        out.t_vals = torch.empty(self.nnz, dtype=torch.float32, device=self.device)
        out.sync_t_vals()
        return out

    @classmethod
    def _k_regular(cls, cols: torch.Tensor) -> "CsrSupport":
        """The pattern whose row n stores the k columns cols[n] ([N, k] int32, ascending in each row), with constant
        zero values, built without a host synchronisation (`k_regular_structure`); `with_values` puts values on it."""
        N, k = cols.shape
        rowptr, col, t_rowptr, t_col, t_perm = k_regular_structure(cols)
        out = cls.__new__(cls)
        out.N, out.rowptr, out.col, out.nnz, out.device = N, rowptr, col, N * k, cols.device
        out.vals = torch.zeros(N * k, dtype=torch.float32, device=cols.device)
        out._t_struct = (t_rowptr, t_col, t_perm)
        out.t_rowptr, out.t_col, out.t_perm = out._t_struct
        out.t_vals = torch.zeros(N * k, dtype=torch.float32, device=cols.device)
        return out

    @classmethod
    def from_dense(cls, G: torch.Tensor) -> "CsrSupport":
        s = G.detach().to_sparse_csr()
        return cls(s.crow_indices(), s.col_indices(), s.values(), G.shape[0])

    @classmethod
    def from_torch_sparse(cls, G: torch.Tensor) -> "CsrSupport":
        s = G.detach().to_sparse_csr()
        return cls(s.crow_indices(), s.col_indices(), s.values(), G.shape[0])

    def to_dense(self) -> torch.Tensor:
        return torch.sparse_csr_tensor(self.rowptr.long(), self.col.long(), self.vals, size=(self.N, self.N)).to_dense()

    def struct(self) -> _lib.StcSupport:
        s = _lib.StcSupport()
        s.kind = _lib.SUPPORT_CSR
        s.nnz = self.nnz
        s.vals, s.rowptr, s.col = self.vals.data_ptr(), self.rowptr.data_ptr(), self.col.data_ptr()
        s.t_vals, s.t_rowptr, s.t_col = self.t_vals.data_ptr(), self.t_rowptr.data_ptr(), self.t_col.data_ptr()
        return s


def k_regular_structure(cols: torch.Tensor):
    """(rowptr, col, t_rowptr, t_col, t_perm) of the pattern storing cols[n] ([N, k] integer, ascending in each row) in
    row n: what `CsrSupport._transpose_structure` gives for the same (rowptr, col), in integer arithmetic on cols'
    device, with no host synchronisation (every size is N or N * k, known on the host).  The keys col * N + row are
    distinct, so the sort needs no stability; the Gs^T row counts come from index_add_ rather than a bincount."""
    N, k = cols.shape
    dev = cols.device
    col = cols.to(torch.int32).reshape(-1).contiguous()
    rowptr = (torch.arange(N + 1, device=dev, dtype=torch.int64) * k).to(torch.int32)
    row = torch.arange(N, device=dev, dtype=torch.int64)[:, None].expand(N, k).reshape(-1)
    colL = col.to(torch.int64)
    t_perm = torch.sort(colL * N + row).indices.contiguous()
    counts = torch.zeros(N, dtype=torch.int64, device=dev).index_add_(0, colL, torch.ones_like(colL))
    t_rowptr = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    t_rowptr[1:] = torch.cumsum(counts, 0)
    return rowptr, col, t_rowptr.to(torch.int32).contiguous(), row[t_perm].to(torch.int32).contiguous(), t_perm


def dense_struct(G: torch.Tensor) -> _lib.StcSupport:
    s = _lib.StcSupport()
    s.kind = _lib.SUPPORT_DENSE
    s.nnz = G.numel()
    s.vals = G.data_ptr()
    return s


def support_apply(Gs, X: torch.Tensor, transpose: bool = True, alpha: float = 1.0, beta: float = 0.0,
                  Z: torch.Tensor = None, out: torch.Tensor = None, rows: torch.Tensor = None) -> torch.Tensor:
    """Y[b,m,...] = alpha * sum_n A(m,n) X[b,n,...] + beta * Z  with A = Gs^T (transpose) or Gs. CUDA only.
    `out` (contiguous, X's shape) receives the result in place of a fresh tensor.  `rows` (int32 CUDA tensor, CSR
    supports only): compute just those output nodes and leave every other row of `out` untouched."""
    lib = _lib.load()
    if not X.is_cuda or X.dtype != torch.float32:
        raise RuntimeError("support_apply needs a float32 CUDA tensor (there is no CPU path)")
    B, N = X.shape[0], X.shape[1]
    Xc = X.contiguous()
    width = Xc[0, 0].numel() if Xc.numel() else 0
    if out is not None:
        if out.shape != Xc.shape or not out.is_contiguous() or out.dtype != torch.float32 or out.device != Xc.device:
            raise RuntimeError("support_apply: `out` must be a contiguous float32 tensor of X's shape on X's device")
        Y = out
    else:
        Y = torch.empty_like(Xc)
    if isinstance(Gs, CsrSupport):
        if transpose:
            Gs.sync_t_vals()
        st = Gs.struct()
        keep = Gs
    else:
        keep = Gs.detach().contiguous()
        st = dense_struct(keep)
    zc = Z.contiguous() if Z is not None else None
    if rows is not None:
        if rows.dtype != torch.int32 or not rows.is_cuda or not rows.is_contiguous():
            raise RuntimeError("support_apply: `rows` must be a contiguous int32 CUDA tensor")
        if out is None:
            raise RuntimeError("support_apply: `rows` needs `out` (the other rows keep their contents)")
        status = lib.stc_support_apply_rows(st, N, B, width, 1 if transpose else 0, Xc.data_ptr(), N * width,
                                            zc.data_ptr() if zc is not None else None, N * width, Y.data_ptr(),
                                            float(alpha), float(beta), rows.data_ptr(), rows.numel(),
                                            torch.cuda.current_stream().cuda_stream)
        _lib.check(status, "stc_support_apply_rows")
        del keep
        return Y
    status = lib.stc_support_apply(st, N, B, width, 1 if transpose else 0, Xc.data_ptr(), N * width,
                                   zc.data_ptr() if zc is not None else None, N * width, Y.data_ptr(),
                                   float(alpha), float(beta), torch.cuda.current_stream().cuda_stream)
    _lib.check(status, "stc_support_apply")
    del keep
    return Y


def support_apply_edge_grad(Gs: CsrSupport, X: torch.Tensor, A: torch.Tensor, dvals: torch.Tensor, coef: float = 1.0,
                            alpha: float = 1.0, beta: float = 0.0, Z: torch.Tensor = None,
                            out: torch.Tensor = None, rows: torch.Tensor = None) -> torch.Tensor:
    """The adjoint hop Y = alpha * Gs X + beta * Z of a CSR support with the gradient of its edge values fused in:
    dvals[e = (n, m)] += coef * sum_{b,...} A[b,n,...] * X[b,m,...]  (dvals [nnz] float32, Gs-CSR order; only added
    to).  Y is what support_apply(Gs, X, transpose=False, ...) returns.  A ([B,N,...] like X) may be a batch-strided
    view whose per-sample slab is contiguous.  `rows` (int32 CUDA tensor; needs `out`): compute just those output
    nodes n, leave every other row of `out` untouched, and add the gradient of those rows' edges only.  CUDA only."""
    lib = _lib.load()
    if not isinstance(Gs, CsrSupport):
        raise RuntimeError("support_apply_edge_grad: CSR supports only (a dense support's gradient is stc_support_outer)")
    for name, t in (("X", X), ("A", A), ("dvals", dvals)):
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"support_apply_edge_grad: {name} must be a float32 CUDA tensor")
    if dvals.shape != (Gs.nnz,) or not dvals.is_contiguous():
        raise RuntimeError(f"support_apply_edge_grad: dvals must be a contiguous [{Gs.nnz}] tensor")
    B, N = X.shape[0], X.shape[1]
    Xc = X.contiguous()
    width = Xc[0, 0].numel() if Xc.numel() else 0
    if A.shape != X.shape:
        raise RuntimeError(f"support_apply_edge_grad: A {tuple(A.shape)} must have X's shape {tuple(X.shape)}")
    Ac = A if (B == 0 or A[0].is_contiguous()) else A.contiguous()
    a_bs = Ac.stride(0) if B > 1 else N * width
    Y = out if out is not None else torch.empty_like(Xc)
    if Y.shape != Xc.shape or not Y.is_contiguous():
        raise RuntimeError("support_apply_edge_grad: `out` must be a contiguous tensor of X's shape")
    zc = Z.contiguous() if Z is not None else None
    common = (Gs.struct(), N, B, width, Xc.data_ptr(), N * width, zc.data_ptr() if zc is not None else None, N * width,
              Y.data_ptr(), float(alpha), float(beta), Ac.data_ptr(), a_bs, float(coef), dvals.data_ptr())
    stream = torch.cuda.current_stream().cuda_stream
    if rows is not None:
        if rows.dtype != torch.int32 or not rows.is_cuda or not rows.is_contiguous():
            raise RuntimeError("support_apply_edge_grad: `rows` must be a contiguous int32 CUDA tensor")
        if out is None:
            raise RuntimeError("support_apply_edge_grad: `rows` needs `out` (the other rows keep their contents)")
        _lib.check(lib.stc_support_apply_rows_edge_grad(*common, rows.data_ptr(), rows.numel(), stream),
                   "stc_support_apply_rows_edge_grad")
        return Y
    _lib.check(lib.stc_support_apply_edge_grad(*common, stream), "stc_support_apply_edge_grad")
    return Y
