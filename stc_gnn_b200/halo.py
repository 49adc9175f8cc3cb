"""Spatial row-partition of a CSR support with per-hop halo exchange (SURVEY.md §8e, BASELINE config 4).

The spatial mode product `Y[b,m,:] = sum_n Gs[n,m] X[b,n,:]` (`framework/STC_GNN.py:37`) is independent per
output node given the features of that node's in-neighbours.  Nodes are split in `world` contiguous blocks
(callers order nodes so that blocks are spatially compact, e.g. Morton / strip order); rank r owns block r of
every [B, N, C, L] tensor.  One Chebyshev hop = exchange the boundary-node slabs (`halo` rows of width B*C*L)
with the ranks that own them, then apply the local operator whose columns are renumbered into
`[local nodes | halo nodes]`.  The categorical mix and the gate contraction are node-local and never communicate.
The adjoint (backward: `dX[b,n,:] = sum_m Gs[n,m] dY[b,m,:]`) is the same scheme on the un-transposed graph; both
directions use one halo set (the union of what either needs) so that forward and backward share buffer layouts.
Parameter gradients are partial sums over a rank's nodes and are all-reduced once per cell backward.

The support's edge values may be learned (values requiring grad, as for `CsrSupport`): the local operators then take
their values from the replicated [nnz] vector through integer maps built once (`PartitionedSupport.maps`), every
adjoint hop also forms the gradient of this rank's edges (`stc_support_apply_rows_edge_grad`, fused into the hop), and
that gradient joins the parameter all-reduce.

Everything here is host logic + `torch.distributed` plumbing (NCCL all-to-all over NVSwitch on the GPU box, gloo in
the CPU tests); the arithmetic is `stc_support_apply` (and its edge-gradient forms) of libstc_b200.so.  There is no CPU arithmetic path: on
non-CUDA tensors `apply` requires the caller to inject `apply_fn` (the tests inject a CPU checker).
"""
from __future__ import annotations

import copy
from dataclasses import dataclass
from typing import Callable, List, Optional

import torch
import torch.distributed as dist

from .dp import shard_bounds


@dataclass
class HaloPlan:
    """Exchange + local operator of ONE direction for ONE rank.

    Operator rows are this rank's output nodes (local numbering 0..nloc-1); its columns index the extended input
    `[local nodes (nloc) | halo nodes (nhalo)]`, halo nodes ordered by owner rank, then by global id.
    """
    rank: int
    world: int
    start: int                      # first global node of this rank's block
    nloc: int
    nhalo: int
    send_idx: List[torch.Tensor]    # per peer: LOCAL indices of the rows this rank sends (sorted by global id)
    recv_counts: List[int]          # per peer: rows received
    halo_global: torch.Tensor       # [nhalo] global ids of the halo nodes, in extended order
    op_row: torch.Tensor            # COO of the local operator: output node (local)
    op_col: torch.Tensor            #                            input node (extended numbering)
    op_val: Optional[torch.Tensor]  # None for a learnable support (its values live in PartitionedSupport.vals)

    @property
    def next(self) -> int:
        return self.nloc + self.nhalo

    @property
    def send_counts(self) -> List[int]:
        return [int(s.numel()) for s in self.send_idx]


def _csr_to_coo(rowptr: torch.Tensor, col: torch.Tensor):
    rowptr = rowptr.long().cpu()
    counts = rowptr[1:] - rowptr[:-1]
    row = torch.repeat_interleave(torch.arange(rowptr.numel() - 1), counts)
    return row, col.long().cpu()


def build_plan(out_idx: torch.Tensor, in_idx: torch.Tensor, vals: Optional[torch.Tensor], num_nodes: int, rank: int,
               world: int, symmetric_halo: bool = False) -> HaloPlan:
    """Plan for the operator `Y[out] += val * X[in]` given as global COO triplets (host tensors; `vals` None: the
    pattern only, as for a learnable support).

    Deterministic and communication-free: every rank derives what each peer needs from the replicated graph.
    `symmetric_halo`: the halo set is the one of the operator AND of its transpose (a superset of what this operator
    reads), so that the plans of both directions share one extended node set -- the backward of the partitioned cell
    runs its adjoint hops on buffers laid out for the forward.  For a structurally symmetric graph nothing is added.
    """
    out_idx, in_idx = out_idx.long().cpu(), in_idx.long().cpu()
    vals = vals.float().cpu() if vals is not None else None
    pair_out, pair_in = (torch.cat([out_idx, in_idx]), torch.cat([in_idx, out_idx])) if symmetric_halo else (out_idx, in_idx)
    bounds = [shard_bounds(num_nodes, p, world) for p in range(world)]
    starts = torch.tensor([b[0] for b in bounds] + [num_nodes])
    owner_of = lambda idx: torch.bucketize(idx, starts[1:], right=True)   # block index of each global node
    out_owner = owner_of(out_idx)
    pair_out_owner, pair_in_owner = owner_of(pair_out), owner_of(pair_in)

    def halo_of(p: int) -> torch.Tensor:   # sorted global ids rank p needs from other ranks
        need = pair_in[(pair_out_owner == p) & (pair_in_owner != p)]
        return torch.unique(need)          # sorted ascending => grouped by owner (blocks are contiguous)

    s, e = bounds[rank]
    my_halo = halo_of(rank)
    my_halo_owner = owner_of(my_halo)
    recv_counts = [int((my_halo_owner == p).sum()) for p in range(world)]
    send_idx = []
    for p in range(world):
        if p == rank:
            send_idx.append(torch.empty(0, dtype=torch.long))
            continue
        hp = halo_of(p)
        send_idx.append(hp[(hp >= s) & (hp < e)] - s)
    mine = out_owner == rank
    r_loc = out_idx[mine] - s
    c_glob = in_idx[mine]
    c_local = (c_glob >= s) & (c_glob < e)
    pos = torch.searchsorted(my_halo, c_glob.clamp(min=0))      # extended slot of halo columns
    c_ext = torch.where(c_local, c_glob - s, (e - s) + pos)
    return HaloPlan(rank=rank, world=world, start=s, nloc=e - s, nhalo=int(my_halo.numel()), send_idx=send_idx,
                    recv_counts=recv_counts, halo_global=my_halo, op_row=r_loc, op_col=c_ext,
                    op_val=vals[mine] if vals is not None else None)


def exchange(plan: HaloPlan, X_local: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """[B, nloc, W] -> [B, nloc + nhalo, W]: append the halo rows received from their owners.

    One all-to-all of packed rows (`[rows, B*W]`, row-major so that split sizes count rows).  With a single rank
    (or no halo anywhere) it degenerates to a copy."""
    B, nloc, W = X_local.shape
    assert nloc == plan.nloc, (nloc, plan.nloc)
    send_rows = [X_local[:, idx.to(X_local.device)].permute(1, 0, 2).reshape(-1, B * W) for idx in plan.send_idx]
    send = torch.cat(send_rows, dim=0).contiguous() if send_rows else X_local.new_empty(0, B * W)
    recv = X_local.new_empty(plan.nhalo, B * W)
    if plan.world > 1:
        dist.all_to_all_single(recv, send, output_split_sizes=plan.recv_counts, input_split_sizes=plan.send_counts,
                               group=group)
    halo = recv.view(plan.nhalo, B, W).permute(1, 0, 2)
    return torch.cat([X_local, halo], dim=1).contiguous()


def exchange_into(plan: HaloPlan, X_ext: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> None:
    """In-place form of `exchange` on an extended tensor [B, nloc + nhalo, W]: only the boundary rows are packed and
    only the halo rows are written (the local block is never copied)."""
    B, next_, W = X_ext.shape
    assert next_ == plan.next, (next_, plan.next)
    if plan.world == 1:     # a property every rank agrees on: with peers, every rank enters the collective below
        return
    send_rows = [X_ext[:, idx.to(X_ext.device)].permute(1, 0, 2).reshape(-1, B * W) for idx in plan.send_idx]
    send = torch.cat(send_rows, dim=0).contiguous() if send_rows else X_ext.new_empty(0, B * W)
    recv = X_ext.new_empty(plan.nhalo, B * W)
    if plan.world > 1:
        dist.all_to_all_single(recv, send, output_split_sizes=plan.recv_counts, input_split_sizes=plan.send_counts,
                               group=group)
    X_ext[:, plan.nloc:] = recv.view(plan.nhalo, B, W).permute(1, 0, 2)


@dataclass
class ValueMaps:
    """Where a rank's local operators take their edge values from, for a learnable support (integer arithmetic, host).

    Both operators are CSR over the extended node set (`next` rows; the halo rows are empty), columns in extended
    numbering, and list the edges of each row in the order the unpartitioned `CsrSupport` walks them, so a hop computes
    bitwise what the unpartitioned hop computes for these rows.
      bwd (operator Gs): rows = this rank's nodes n, edges in global Gs-CSR order.  Its values are the slice
          vals[edge_lo:edge_hi] and its edge gradient is the same slice of the global [nnz] gradient.
      fwd (operator Gs^T): rows = this rank's nodes m, edges sorted by (m, global n) as in `CsrSupport.t_perm`; edge i
          is global edge fwd_ids[i], so its values are vals[fwd_ids].
    Gather layout of an [nnz] vector whose slices [edge_lo:edge_hi] live on their ranks (`gather_edges`): every rank's
    slice is padded to `edge_pad` floats, so rank r's slice lands at [r * edge_pad, r * edge_pad + hi_r - lo_r) of the
    all-gathered buffer; `edge_bounds[r]` = (lo_r, hi_r)."""
    edge_lo: int
    edge_hi: int
    bwd_rowptr: torch.Tensor
    bwd_col: torch.Tensor
    fwd_rowptr: torch.Tensor
    fwd_col: torch.Tensor
    fwd_ids: torch.Tensor
    edge_bounds: List[tuple]
    edge_pad: int

    def padded_index(self, ids: torch.Tensor) -> torch.Tensor:
        """Positions in the padded all-gather buffer of the global edges `ids` (integer arithmetic on ids' device, no
        host copy)."""
        out = ids.clone()
        for r, (lo, hi) in enumerate(self.edge_bounds):
            out = torch.where((ids >= lo) & (ids < hi), ids + (r * self.edge_pad - lo), out)
        return out


def _csr_operator(rowptr: torch.Tensor, col: torch.Tensor, vals: torch.Tensor, n: int):
    """A CsrSupport whose Gs IS the given [n, n] operator; it is only ever applied with transpose=False, so its Gs^T
    fields alias Gs instead of holding a transpose nobody walks."""
    from .support import CsrSupport
    sup = CsrSupport.__new__(CsrSupport)
    sup.N, sup.rowptr, sup.col, sup.vals = n, rowptr, col, vals
    sup.nnz, sup.device = int(vals.numel()), vals.device
    sup.t_rowptr, sup.t_col, sup.t_vals = rowptr, col, vals
    sup.t_perm, sup._t_struct = None, None
    return sup


class PartitionedSupport:
    """A CSR spatial support `Gs` [N, N] row-partitioned over `world` ranks.

    `rowptr, col, vals` is the GLOBAL `Gs` in CSR (replicated; N = 65,536, nnz ~ 0.6 M is 7 MB).  The pattern may
    live on the host or the device.  `fwd` is the plan of the forward mode product (operator Gs^T: output m, input n
    for every stored Gs[n,m]), `bwd` the plan of its adjoint (operator Gs).

    Constant support: `vals` does not require grad; the local operators are built from it once.
    Learnable support: `vals` requires grad (an `nn.Parameter` [nnz] in Gs-CSR order, or values computed from one,
    e.g. `softplus(raw)`, see `with_values`).  The pattern is fixed and every stored edge is trainable, including
    edges stored as 0.  The local operators take their values from `vals` through `maps()`: the adjoint operator uses
    the view vals[edge_lo:edge_hi], the forward operator a persistent buffer that one gather refreshes before every
    partitioned cell forward, so an in-place optimizer update is seen by the next step.  The cell returns the
    gradient of `vals` ([nnz], Gs-CSR order).  The values must be identical on every rank: a rank only reads the
    edges of its own rows, so ranks holding different values would silently mix them.
    """

    def __init__(self, rowptr: torch.Tensor, col: torch.Tensor, vals: torch.Tensor, num_nodes: int, rank: int,
                 world: int, group: Optional[dist.ProcessGroup] = None):
        n_idx, m_idx = _csr_to_coo(rowptr, col)      # Gs[n, m]
        self.N, self.rank, self.world, self.group = int(num_nodes), rank, world, group
        self._rowptr, self._col = rowptr.long().cpu(), m_idx
        self.nnz = int(m_idx.numel())
        self.vals = self._check_values(vals) if vals.requires_grad else None
        plan_vals = None if self.vals is not None else vals
        # one extended node set [local | halo] for both directions (see build_plan)
        self.fwd = build_plan(m_idx, n_idx, plan_vals, num_nodes, rank, world, symmetric_halo=True)
        self.bwd = build_plan(n_idx, m_idx, plan_vals, num_nodes, rank, world, symmetric_halo=True)
        assert self.fwd.nhalo == self.bwd.nhalo and torch.equal(self.fwd.halo_global, self.bwd.halo_global)
        self.start, self.nloc = self.fwd.start, self.fwd.nloc
        # STC_Cell / RecurrentStack accept this object as `Gs` (blocks in, blocks out).  True: every cell backward
        # all-reduces its parameter gradients; False: the caller reduces once per step (dp.allreduce_gradients).
        self.reduce_per_cell = True
        self._dev = {}       # structure on the device (shared with `with_values` copies)
        self._ops = {}       # learnable: the local operators bound to this object's `vals`
        self._streams = {}   # side streams and events of the exchange overlap (a RowPartition shares its own)

    @classmethod
    def from_dense(cls, G: torch.Tensor, rank: int, world: int, group=None) -> "PartitionedSupport":
        s = G.detach().cpu().to_sparse_csr()
        return cls(s.crow_indices(), s.col_indices(), s.values(), G.shape[0], rank, world, group)

    @classmethod
    def from_csr_support(cls, cs, rank: int, world: int, group=None) -> "PartitionedSupport":
        """The partition of a `CsrSupport`; a learnable one shares its `vals` (the same tensor, not a copy)."""
        if getattr(cs, "batch", None) is not None:
            raise RuntimeError("PartitionedSupport.from_csr_support: per-sample edge values [B, nnz] are not supported "
                               "on the row-partitioned graph (one set of values is shared by the batch)")
        return cls(cs.rowptr, cs.col, cs.vals, cs.N, rank, world, group)

    @classmethod
    def k_regular(cls, cols: torch.Tensor, rank: int, world: int, group=None) -> "PartitionedSupport":
        """The partition of the k-regular pattern whose row n stores the columns cols[n] ([N, k] integer, ascending in
        each row, identical on every rank), with constant zero values: field for field what
        `PartitionedSupport(k * arange(N + 1), cols.flatten(), zeros, N, rank, world, group)` builds (plans, `maps()`
        and the exchange state), computed in integer torch ops on cols' device (CPU or CUDA) with one device-to-host
        copy of a few counts.  `RowPartition.support` is the same with the partition's persistent state."""
        return RowPartition(cols.shape[0], rank, world, group).support(cols)

    @property
    def learnable(self) -> bool:
        """True when the local operators take their values from `vals` (see the class docstring); the cell returns
        the gradient of `vals` when it requires grad."""
        return self.vals is not None

    def _check_values(self, vals: torch.Tensor) -> torch.Tensor:
        if vals.dim() == 2:
            raise RuntimeError(f"PartitionedSupport: per-sample edge values {tuple(vals.shape)} are not supported on the "
                               f"row-partitioned graph; give one [nnz] vector (nnz = {self.nnz}) shared by the batch")
        if vals.dim() != 1 or vals.numel() != self.nnz:
            raise RuntimeError(f"PartitionedSupport: edge values must be a [nnz] vector in Gs-CSR order "
                               f"(nnz = {self.nnz}), got shape {tuple(vals.shape)}")
        return vals

    def with_values(self, vals: torch.Tensor) -> "PartitionedSupport":
        """A learnable support with this one's pattern, plans and maps and new edge values [nnz] (Gs-CSR order)."""
        out = copy.copy(self)
        out.vals = self._check_values(vals)
        out._ops = {}
        return out

    def maps(self) -> ValueMaps:
        """The value maps of this rank's local operators (computed once per pattern, in integer arithmetic)."""
        m = self._dev.get("maps")
        if m is None:
            rowptr, col, N = self._rowptr, self._col, self.N
            s, e, nloc, nhalo = self.start, self.start + self.nloc, self.nloc, self.fwd.nhalo
            halo = self.fwd.halo_global
            ext = lambda c: torch.where((c >= s) & (c < e), c - s, nloc + torch.searchsorted(halo, c))
            lo, hi = int(rowptr[s]), int(rowptr[e])
            pad = lambda rp: torch.cat([rp, rp[-1:].expand(nhalo)])
            row = torch.repeat_interleave(torch.arange(N), rowptr[1:] - rowptr[:-1], output_size=self.nnz)
            mine = torch.nonzero((col >= s) & (col < e)).flatten()           # edges (n, m) with m on this rank
            ids = mine[torch.sort((col[mine] - s) * N + row[mine], stable=True).indices]
            f_rowptr = torch.zeros(nloc + 1, dtype=torch.long)
            f_rowptr[1:] = torch.cumsum(torch.bincount(col[ids] - s, minlength=nloc), 0)
            bounds = [(int(rowptr[a]), int(rowptr[b])) for a, b in (shard_bounds(N, r, self.world)
                                                                    for r in range(self.world))]
            m = self._dev["maps"] = ValueMaps(edge_lo=lo, edge_hi=hi, bwd_rowptr=pad(rowptr[s:e + 1] - lo),
                                              bwd_col=ext(col[lo:hi]), fwd_rowptr=pad(f_rowptr), fwd_col=ext(row[ids]),
                                              fwd_ids=ids, edge_bounds=bounds,
                                              edge_pad=max(b - a for a, b in bounds))
        return m

    def sync_values(self, device) -> None:
        """Learnable: gather the forward operator's values from `vals`, on the current stream."""
        if self.learnable:
            op, ids = self._learned_operator("fwd", device)
            torch.index_select(self.vals.detach(), 0, ids, out=op.vals)

    def local_slice(self, X: torch.Tensor, node_dim: int = 1) -> torch.Tensor:
        """This rank's node block of a global tensor."""
        return X.narrow(node_dim, self.start, self.nloc)

    # -- device form of the local operators (square, padded with empty rows so the square C-ABI kernel applies) --
    def _operator_structure(self, direction: str, device):
        """(rowptr, col, forward map or None) of the local operator of `direction` (see ValueMaps), on the device."""
        skey = ("learned", direction, str(device))
        st = self._dev.get(skey)
        if st is None:
            m = self.maps()
            rp, c = (m.fwd_rowptr, m.fwd_col) if direction == "fwd" else (m.bwd_rowptr, m.bwd_col)
            ids = m.fwd_ids.to(device) if direction == "fwd" else None
            st = self._dev[skey] = (rp.to(torch.int32).to(device), c.to(torch.int32).to(device), ids)
        return st

    def local_operator(self, direction: str, vals: torch.Tensor):
        """The local operator of `direction` (see ValueMaps) carrying `vals` (float32, on the device: 'bwd' the
        [edge_hi - edge_lo] edges of this rank's rows in Gs-CSR order, 'fwd' the edges fwd_ids), as a CsrSupport that
        is applied with transpose=False over the extended node set.  Only the pattern is read when it is handed to the
        generator's kernels."""
        rp, c, _ = self._operator_structure(direction, vals.device)
        return _csr_operator(rp, c, vals, self.fwd.next)

    def _learned_operator(self, direction: str, device):
        """(local operator bound to `vals`, forward map on the device or None)."""
        key = (direction, str(device))
        hit = self._ops.get(key)
        if hit is None:
            m = self.maps()
            rp, c, ids = self._operator_structure(direction, device)
            v = self.vals.detach()
            if not v.is_cuda or v.dtype != torch.float32 or not v.is_contiguous() or v.device != torch.device(device):
                raise RuntimeError(f"PartitionedSupport: learnable values must be a contiguous float32 tensor on {device}, "
                                   f"got {v.dtype} on {v.device}")
            vals = torch.empty(ids.numel(), dtype=torch.float32, device=device) if ids is not None else \
                v[m.edge_lo:m.edge_hi]
            hit = self._ops[key] = (_csr_operator(rp, c, vals, self.fwd.next), ids)
        return hit

    def device_support(self, direction: str, device):
        """CsrSupport G_loc with `support_apply(G_loc, X_ext, transpose=self.transposed(direction))[:, :nloc]` ==
        operator.  Learnable: G_loc IS the operator, bound to `vals` (call `sync_values` before a forward hop)."""
        if self.learnable:
            return self._learned_operator(direction, device)[0]
        key = (direction, str(device))
        if key not in self._dev:
            from .support import CsrSupport
            plan = self.fwd if direction == "fwd" else self.bwd
            n = plan.next
            # fwd: operator A_f[m_loc, n_ext] is applied as G_loc^T with G_loc[n_ext, m_loc]; bwd: G_loc = A_b
            r, c = (plan.op_col, plan.op_row) if direction == "fwd" else (plan.op_row, plan.op_col)
            g = torch.sparse_coo_tensor(torch.stack([r, c]), plan.op_val, size=(n, n)).coalesce().to_sparse_csr()
            self._dev[key] = CsrSupport(g.crow_indices().to(device), g.col_indices().to(device),
                                        g.values().to(device), n)
        return self._dev[key]

    def transposed(self, direction: str) -> bool:
        """The `transpose` flag `device_support(direction)` is applied with."""
        return direction == "fwd" and not self.learnable

    def apply(self, X_local: torch.Tensor, direction: str = "fwd", alpha: float = 1.0, beta: float = 0.0,
              Z_local: Optional[torch.Tensor] = None,
              apply_fn: Optional[Callable[[HaloPlan, torch.Tensor], torch.Tensor]] = None) -> torch.Tensor:
        """One hop on this rank's block: `alpha * A X + beta * Z`, A = Gs^T ('fwd') or Gs ('bwd').

        X_local, Z_local: [B, nloc, ...feature axes]; returns the same shape.  `apply_fn(plan, X_ext) -> [B, nloc, W]`
        replaces the CUDA kernel (tests inject a CPU checker; there is no built-in CPU arithmetic)."""
        plan = self.fwd if direction == "fwd" else self.bwd
        shape = X_local.shape
        B = shape[0]
        X3 = X_local.reshape(B, plan.nloc, -1)
        X_ext = exchange(plan, X3, self.group)
        if apply_fn is not None:
            Y = apply_fn(plan, X_ext)
            Y = alpha * Y + (beta * Z_local.reshape(B, plan.nloc, -1) if beta != 0.0 else 0.0)
            return Y.reshape(shape)
        if not X_local.is_cuda:
            raise RuntimeError("PartitionedSupport.apply needs CUDA tensors (there is no CPU path)")
        from .support import support_apply
        Z_ext = None
        if beta != 0.0:
            Z3 = Z_local.reshape(B, plan.nloc, -1)
            Z_ext = torch.cat([Z3, Z3.new_zeros(B, plan.nhalo, Z3.shape[-1])], dim=1)
        if direction == "fwd":
            self.sync_values(X_local.device)
        Y_ext = support_apply(self.device_support(direction, X_local.device), X_ext, transpose=self.transposed(direction),
                              alpha=alpha, beta=beta, Z=Z_ext)
        return Y_ext[:, :plan.nloc].reshape(shape)

    # -- device-side exchange state: packed index lists, interior / boundary row lists, persistent buffers --
    def _device_state(self, direction: str, device):
        key = ("xchg", direction, str(device))
        st = self._dev.get(key)
        if st is None:
            plan = self.fwd if direction == "fwd" else self.bwd
            send = torch.cat(plan.send_idx) if plan.send_idx else torch.empty(0, dtype=torch.long)
            has_halo_col = torch.zeros(plan.nloc, dtype=torch.bool)
            has_halo_col[plan.op_row[plan.op_col >= plan.nloc]] = True
            interior = torch.nonzero(~has_halo_col).flatten()
            # boundary pass: local rows that read a halo column + the halo rows themselves (empty operator rows: they
            # come out as beta * Z, i.e. finite -- the node-local stages run over the extended node set)
            boundary = torch.cat([torch.nonzero(has_halo_col).flatten(), torch.arange(plan.nloc, plan.next)])
            st = self._dev[key] = {
                "send_idx": send.to(torch.int32).to(device), "nsend": int(send.numel()),
                "interior": interior.to(torch.int32).to(device), "boundary": boundary.to(torch.int32).to(device),
                "buffers": {},
            }
        return st

    def _stream_state(self, direction: str, device):
        """(side stream, ready event, done event) of the exchange overlap of `direction`, created once per partition."""
        key = (direction, str(device))
        ss = self._streams.get(key)
        if ss is None:
            ss = self._streams[key] = (torch.cuda.Stream(device=device), torch.cuda.Event(), torch.cuda.Event())
        return ss

    def _buffers(self, st, plan, slab: int, device):
        buf = st["buffers"].get(slab)
        if buf is None:
            if len(st["buffers"]) > 4:
                st["buffers"].clear()
            buf = st["buffers"][slab] = (torch.empty(st["nsend"], slab, dtype=torch.float32, device=device),
                                         torch.empty(plan.nhalo, slab, dtype=torch.float32, device=device))
        return buf

    def hop_ext(self, X_ext: torch.Tensor, out_ext: torch.Tensor, Z_ext: Optional[torch.Tensor] = None,
                alpha: float = 1.0, beta: float = 0.0, direction: str = "fwd", *, A_ext: Optional[torch.Tensor] = None,
                coef: float = 1.0, dvals: Optional[torch.Tensor] = None) -> None:
        """One hop on EXTENDED tensors [B, nloc + nhalo, ...] (CUDA): `out_ext = alpha * A X_ext + beta * Z_ext` with the
        local operator (square over the extended index set; the halo nodes have empty operator rows).

        The halo rows of `X_ext` are refreshed in place from their owners ON A SIDE STREAM -- `stc_halo_pack` of the
        boundary rows into a persistent send buffer, one NCCL all-to-all of packed rows, `stc_halo_unpack` into the halo
        rows -- while the main stream already computes the INTERIOR output rows (those whose neighbours are all local,
        `stc_support_apply_rows`); the main stream then waits for the exchange and computes the boundary rows.  No
        tensor is copied, sliced or allocated per hop (`_overlapped`).

        Edge-gradient form (learnable support, direction 'bwd'): `dvals` is this rank's slice
        [edge_lo:edge_hi] of the global [nnz] gradient, and both launches also add
        dvals[e = (n, m)] += coef * sum A_ext[:, n] * X_ext[:, m]  (A_ext [B, nloc + nhalo, ...] the forward term the hop's
        adjoint belongs to; read at the local rows only).  A learnable forward hop reads the values `sync_values` last
        gathered."""
        from .support import support_apply, support_apply_edge_grad
        plan = self.fwd if direction == "fwd" else self.bwd
        B = X_ext.shape[0]
        X3 = X_ext.view(B, plan.next, -1)
        out3 = out_ext.view(B, plan.next, -1)
        Z3 = None if Z_ext is None else Z_ext.view(B, plan.next, -1)
        sup = self.device_support(direction, X_ext.device)
        if dvals is not None:
            if direction != "bwd" or not self.learnable or A_ext is None:
                raise RuntimeError("hop_ext: an edge gradient needs a learnable support, direction 'bwd' and A_ext")
            A3 = A_ext.view(B, plan.next, -1)
            hop = lambda rows=None: support_apply_edge_grad(sup, X3, A3, dvals, coef=coef, alpha=alpha, beta=beta, Z=Z3,
                                                            out=out3, rows=rows)
        else:
            tr = self.transposed(direction)
            hop = lambda rows=None: support_apply(sup, X3, transpose=tr, alpha=alpha, beta=beta, Z=Z3, out=out3, rows=rows)
        self._overlapped(direction, X3, hop)

    def _overlapped(self, direction: str, X3: torch.Tensor, launch: Callable[[Optional[torch.Tensor]], None]) -> None:
        """The exchange-overlap skeleton of every computation on an extended tensor X3 [B, nloc + nhalo, W] whose output
        rows read their neighbours' rows of X3 through the local operator of `direction`.

        The halo rows of X3 are refreshed in place ON A SIDE STREAM -- `stc_halo_pack` of the boundary rows into a
        persistent send buffer, one all-to-all of packed rows, `stc_halo_unpack` into the halo rows -- while the main
        stream runs `launch(interior rows)` (the rows whose neighbours are all local); the main stream then waits for
        the exchange and runs `launch(boundary rows)` (the rows reading a halo row, and the halo rows).  The row lists
        are int32 device tensors.  At world 1 it is `launch(None)`: every row, nothing exchanged."""
        from . import _lib
        plan = self.fwd if direction == "fwd" else self.bwd
        if plan.world == 1:
            launch(None)
            return
        B, _, W = X3.shape
        lib = _lib.load()
        st = self._device_state(direction, X3.device)
        send, recv = self._buffers(st, plan, B * W, X3.device)
        side, ready, done = self._stream_state(direction, X3.device)
        main = torch.cuda.current_stream()
        ready.record(main)                           # X3's local rows are final once the main stream gets here
        with torch.cuda.stream(side):
            side.wait_event(ready)
            _lib.check(lib.stc_halo_pack(X3.data_ptr(), plan.next * W, W, B, st["send_idx"].data_ptr(), st["nsend"],
                                         send.data_ptr(), side.cuda_stream), "stc_halo_pack")
            dist.all_to_all_single(recv, send, output_split_sizes=plan.recv_counts, input_split_sizes=plan.send_counts,
                                   group=self.group)
            _lib.check(lib.stc_halo_unpack(recv.data_ptr(), W, B, plan.nloc, plan.nhalo, X3.data_ptr(), plan.next * W,
                                           side.cuda_stream), "stc_halo_unpack")
            done.record(side)
        if st["interior"].numel():
            launch(st["interior"])
        main.wait_event(done)
        launch(st["boundary"])

    def spatial_terms(self, X_local: torch.Tensor, Ks: int, apply_fn=None) -> List[torch.Tensor]:
        """Feature-side Chebyshev terms Y_0..Y_{Ks-1} of this rank's block (Y_1 = Gs^T Y_0, Y_k = 2 Gs^T Y_{k-1} - Y_{k-2};
        `framework/STC_GNN.py:24-29` applied on the feature side): Ks-1 hops, one halo exchange each."""
        terms = [X_local]
        for k in range(1, Ks):
            if k == 1:
                terms.append(self.apply(terms[0], "fwd", apply_fn=apply_fn))
            else:
                terms.append(self.apply(terms[k - 1], "fwd", alpha=2.0, beta=-1.0, Z_local=terms[k - 2], apply_fn=apply_fn))
        return terms


def _positions(mask: torch.Tensor, count: int) -> torch.Tensor:
    """The indices of the True entries of a 1-D mask, ascending; `count` (known on the host) of them.  A stable sort of
    the inverted mask instead of `nonzero`, which would synchronise with the device."""
    return torch.sort((~mask).to(torch.int8), stable=True).indices[:count]


class RowPartition:
    """The row partition of an N-node graph over `world` ranks (rank r owns the nodes `dp.shard_bounds(N, r, world)`)
    without a fixed pattern: the generator selects a new pattern on every forward (`SparseGraphGenerator(...)(X_seq,
    k=k, partition=...)`) and `support(cols)` partitions it on the device.  The state that outlives a pattern lives
    here: the side streams and events of the exchange overlap, and `reduce_per_cell` (copied onto every support; see
    `PartitionedSupport`)."""

    def __init__(self, num_nodes: int, rank: int, world: int, group: Optional[dist.ProcessGroup] = None):
        self.N, self.rank, self.world, self.group = int(num_nodes), rank, world, group
        self.start, stop = shard_bounds(self.N, rank, world)
        self.nloc = stop - self.start
        self.reduce_per_cell = True
        self._streams = {}

    def gather_rows(self, x_loc: torch.Tensor) -> torch.Tensor:
        """[N, ...] from every rank's node block x_loc [nloc, ...] (one all-gather; the blocks are padded to the largest,
        ceil(N / world) rows, and compacted); x_loc itself at world 1.  Every rank must call it."""
        if self.world == 1:
            return x_loc
        big = shard_bounds(self.N, 0, self.world)[1]
        send = x_loc.new_zeros((big,) + tuple(x_loc.shape[1:]))
        send[:self.nloc] = x_loc
        out = x_loc.new_empty((self.world * big,) + tuple(x_loc.shape[1:]))
        dist.all_gather_into_tensor(out, send, group=self.group)
        return torch.cat([out.narrow(0, r * big, e - s) for r, (s, e) in
                          enumerate(shard_bounds(self.N, r, self.world) for r in range(self.world))])

    def support(self, cols: torch.Tensor) -> PartitionedSupport:
        """`PartitionedSupport.k_regular(cols, rank, world, group)` sharing this partition's streams and events.

        Every rank derives what each peer needs from the replicated selection (as `build_plan` does from the replicated
        graph), in integer torch ops on cols' device.  The halo of rank p is the set of nodes outside block p that a row
        of p reads or that reads a row of p (the symmetric halo); it is held as a [world, N] membership table, from which
        the halo lists, the send lists, the extended column numbering and the per-peer counts follow by cumulative
        sums.  The Gs^T side comes from `support.k_regular_structure`.  One device-to-host copy carries the sizes the
        host needs (nhalo, the per-peer send and receive counts, the interior counts of both directions, the range of
        this rank's columns in Gs^T order)."""
        from .support import k_regular_structure
        N, k = cols.shape
        if N != self.N:
            raise RuntimeError(f"RowPartition: the selection has {N} rows, the partition {self.N} nodes")
        dev, L = cols.device, torch.long
        rank, world, s, nloc = self.rank, self.world, self.start, self.nloc
        e = s + nloc
        rowptr, col32, t_rowptr, t_col, t_perm = k_regular_structure(cols)
        col, nnz = col32.to(L), N * k
        row = torch.arange(N, device=dev, dtype=L)[:, None].expand(N, k).reshape(-1)
        base, extra = divmod(N, world)
        p = torch.arange(world + 1, device=dev, dtype=L)
        starts = p * base + p.clamp(max=extra)                     # shard_bounds of every rank, then N
        owner = lambda x: torch.bucketize(x, starts[1:], right=True)
        ro, co = owner(row), owner(col)
        cross = (ro != co).to(L)
        member = torch.zeros(world * N, dtype=L, device=dev)
        member.index_add_(0, ro * N + col, cross).index_add_(0, co * N + row, cross)
        member = (member > 0).view(world, N)                       # member[p, x]: x is in the halo of rank p
        mine = member[rank]
        csum = torch.zeros(N + 1, dtype=L, device=dev)
        csum[1:] = torch.cumsum(mine, 0)
        recv = csum[starts[1:]] - csum[starts[:-1]]
        sendm = member[:, s:e]                                     # what each peer needs of this rank's nodes
        send = sendm.sum(1)
        ids = torch.arange(N, device=dev, dtype=L)
        ext = torch.where((ids >= s) & (ids < e), ids - s, nloc + csum[1:] - 1)   # extended numbering of halo + local
        own = co.view(N, k)[s:e] != rank
        has_b = own.any(1)                                         # adjoint rows reading a halo column
        has_f = torch.zeros(nloc, dtype=L, device=dev)
        if nloc:
            into = ((co == rank) & (ro != rank)).to(L)
            has_f.index_add_(0, torch.where(co == rank, col - s, 0), into)
        has_f = has_f > 0                                          # forward rows reading a halo column
        info = torch.cat([csum[N:], recv, send, (~has_f).sum().view(1), (~has_b).sum().view(1),
                          t_rowptr[s:s + 1].to(L), t_rowptr[e:e + 1].to(L)]).cpu().tolist()   # the one host copy
        nhalo, recv_counts, send_counts = info[0], info[1:1 + world], info[1 + world:1 + 2 * world]
        nint_f, nint_b, f0, f1 = info[1 + 2 * world:]
        halo_global = _positions(mine, nhalo)
        send_cat = _positions(sendm.reshape(-1), sum(send_counts)) % max(nloc, 1)
        send_idx = list(torch.split(send_cat, send_counts))
        lo, hi = k * s, k * e
        fwd_ids = t_perm[f0:f1]                                    # this rank's columns, Gs^T order = (m, global n)
        f_edges = torch.sort(fwd_ids).values                       # the same edges in Gs-CSR order
        zeros = lambda n: torch.zeros(n, dtype=torch.float32, device=dev)

        def plan(op_row, op_col):
            return HaloPlan(rank=rank, world=world, start=s, nloc=nloc, nhalo=nhalo, send_idx=send_idx,
                            recv_counts=recv_counts, halo_global=halo_global, op_row=op_row, op_col=op_col,
                            op_val=zeros(op_row.numel()))

        ps = PartitionedSupport.__new__(PartitionedSupport)
        ps.N, ps.rank, ps.world, ps.group = N, rank, world, self.group
        ps._rowptr, ps._col, ps.nnz, ps.vals = rowptr.to(L), col, nnz, None
        ps.fwd = plan(col[f_edges] - s, ext[row[f_edges]])
        ps.bwd = plan(row[lo:hi] - s, ext[col[lo:hi]])
        ps.start, ps.nloc = s, nloc
        ps.reduce_per_cell = self.reduce_per_cell
        ps._ops, ps._streams = {}, self._streams
        nxt = nloc + nhalo
        pad = lambda rp: torch.cat([rp, rp[-1:].expand(nhalo)])
        bounds = [(k * a, k * b) for a, b in (shard_bounds(N, r, world) for r in range(world))]
        maps = ValueMaps(edge_lo=lo, edge_hi=hi, bwd_rowptr=pad(rowptr[s:e + 1].to(L) - lo), bwd_col=ps.bwd.op_col,
                         fwd_rowptr=pad(t_rowptr[s:e + 1].to(L) - f0), fwd_col=ext[t_col[f0:f1].to(L)], fwd_ids=fwd_ids,
                         edge_bounds=bounds, edge_pad=max(b - a for a, b in bounds))
        ps._dev = {"maps": maps}
        halo_rows = torch.arange(nloc, nxt, device=dev, dtype=L)
        for direction, has, nint in (("fwd", has_f, nint_f), ("bwd", has_b, nint_b)):
            ps._dev[("xchg", direction, str(dev))] = {
                "send_idx": send_cat.to(torch.int32), "nsend": int(send_cat.numel()),
                "interior": _positions(~has, nint).to(torch.int32),
                "boundary": torch.cat([_positions(has, nloc - nint), halo_rows]).to(torch.int32), "buffers": {}}
        return ps


def adjoint_chain_ext(ps: PartitionedSupport, ybar: List[torch.Tensor], hop: Optional[Callable] = None,
                      terms: Optional[List[torch.Tensor]] = None, dvals: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Reverse of the feature-side recurrence (Y_1 = Gs^T Y_0, Y_k = 2 Gs^T Y_{k-1} - Y_{k-2}) on EXTENDED adjoints.

    `ybar[k]` [B, nloc + nhalo, ...] holds dL/dY_k of this rank's nodes in its local rows (halo rows: anything).  In
    place, for k = Ks-1 .. 1:  ybar[k-1] += (2 if k >= 2 else 1) * Gs ybar[k]  (one halo exchange of ybar[k], adjoint
    plan) and ybar[k-2] -= ybar[k] (local rows only).  Returns ybar[0], whose local rows are dL/dY_0.
    `terms` (forward terms Y_0 .. Y_{Ks-2}, extended) and `dvals` (this rank's slice of the [nnz] edge gradient of a
    learnable support): every hop also adds the same coefficient times Y_{k-1} (x) ybar[k] at this rank's edges.
    `hop(X_ext, out_ext, Z_ext, alpha, beta, direction)` replaces `ps.hop_ext` (the CPU tests inject a checker); with
    `dvals` it is also passed `A_ext=`, `coef=` and `dvals=` as keywords."""
    hop = hop or (lambda X, out, Z, alpha, beta, direction, **eg: ps.hop_ext(X, out, Z_ext=Z, alpha=alpha, beta=beta,
                                                                            direction=direction, **eg))
    n = ps.nloc
    for k in range(len(ybar) - 1, 0, -1):
        coef = 2.0 if k >= 2 else 1.0
        if dvals is None:
            hop(ybar[k], ybar[k - 1], ybar[k - 1], coef, 1.0, "bwd")
        else:
            hop(ybar[k], ybar[k - 1], ybar[k - 1], coef, 1.0, "bwd", A_ext=terms[k - 1], coef=coef, dvals=dvals)
        if k >= 2:
            ybar[k - 2][:, :n].sub_(ybar[k][:, :n])
    return ybar[0]


def gather_edges_padded(ps: PartitionedSupport, x_loc: torch.Tensor, async_op: bool = False):
    """All-gather of every rank's slice x_loc [edge_hi - edge_lo] of an [nnz] edge vector (Gs-CSR order) into the padded
    buffer [world * edge_pad] of `ValueMaps` (one collective: NCCL needs equal chunks, so each slice is padded to the
    largest).  Returns (buffer, work handle or None); the padding entries are zeros.  World > 1 only."""
    m = ps.maps()
    send = x_loc.new_zeros(m.edge_pad)
    send[:x_loc.numel()] = x_loc
    out = x_loc.new_empty(ps.world * m.edge_pad)
    work = dist.all_gather_into_tensor(out, send, group=ps.group, async_op=async_op)
    return out, work


def unpad_edges(ps: PartitionedSupport, buf: torch.Tensor) -> torch.Tensor:
    """The [nnz] vector (Gs-CSR order) of a padded all-gather buffer."""
    m = ps.maps()
    return torch.cat([buf.narrow(0, r * m.edge_pad, hi - lo) for r, (lo, hi) in enumerate(m.edge_bounds)])


class _GatherEdges(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_loc, ps):
        m = ps.maps()
        ctx.lo, ctx.n = m.edge_lo, m.edge_hi - m.edge_lo
        return unpad_edges(ps, gather_edges_padded(ps, x_loc.detach().contiguous())[0])

    @staticmethod
    def backward(ctx, dfull):
        return dfull.narrow(0, ctx.lo, ctx.n), None


def gather_edges(ps: PartitionedSupport, x_loc: torch.Tensor) -> torch.Tensor:
    """The full [nnz] edge vector (Gs-CSR order, the same bytes on every rank) from every rank's slice
    x_loc = full[edge_lo:edge_hi], in one all-gather (`gather_edges_padded`); x_loc itself at world 1.

    Differentiable, with NO communication in the backward: the gradient of x_loc is the slice [edge_lo:edge_hi] of the
    gradient arriving at the full vector, which must therefore be exact on this rank's edges.  A partitioned cell
    guarantees that for the learnable support it returns: with `reduce_per_cell` the [nnz] gradient is all-reduced,
    without it this rank's partial gradient is non-zero only in its own slice and complete there (a rank's adjoint
    hops form the gradient of the edges of its own rows, and of no other)."""
    if ps.world == 1:
        return x_loc
    return _GatherEdges.apply(x_loc, ps)


def _partitioned_forward(Gc, Xt, Ht_1, Wg, bg, Wc, bc, cfg, fwd_only):
    """The forward of one STC cell on this rank's node block: the node-local stages (`stc_cell_fwd_stage`, or
    `stc_cell_fwd_only_stage` on the smaller forward-only workspace with `fwd_only`) with the spatial hops in between.
    Returns (the local block of H', (Gc, Xe, He, Wg, Wc, buffer) as the stages read them, dims, buffer layout)."""
    from . import _lib
    from .cell import _activation_code, _ptr
    ps, Ks, Kc, activation, reduce_params = cfg
    lib = _lib.load()
    ps.sync_values(Xt.device)        # learnable: the values as they are now (e.g. after an optimizer step)
    B, n, C, Din = Xt.shape
    h = Ht_1.shape[-1]
    # Everything lives in the EXTENDED node set [local | halo]: the node-local stages simply run over
    # nloc + nhalo nodes (the halo rows, ~1 % at k = 8, are recomputed garbage that the next exchange overwrites),
    # so the spatial terms are written straight into the `saved` regions the stages read -- no slicing, no compaction.
    ne = ps.fwd.next
    Gc = Gc.detach().contiguous()
    Wg, Wc = Wg.detach().contiguous(), Wc.detach().contiguous()
    bg = bg.detach().contiguous() if bg is not None else None
    bc = bc.detach().contiguous() if bc is not None else None
    Xe = Xt.new_zeros(B, ne, C, Din)
    Xe[:, :n] = Xt.detach()
    He = Ht_1.new_zeros(B, ne, C, h)
    He[:, :n] = Ht_1.detach()
    dims = _lib.StcDims(B, ne, C, Din, h, Ks, Kc, _activation_code(activation), 1 if bg is not None else 0)
    lay = _lib.saved_layout(dims, fwd_only)
    nbytes = lib.stc_cell_fwd_only_bytes(dims) if fwd_only else lib.stc_cell_saved_bytes(dims)
    saved = torch.empty(nbytes // 4, dtype=torch.float32, device=Xt.device)
    Hn = torch.empty_like(He)
    R = B * ne * C
    stream = torch.cuda.current_stream().cuda_stream
    run_stage, what = ((lib.stc_cell_fwd_only_stage, "stc_cell_fwd_only_stage") if fwd_only else
                       (lib.stc_cell_fwd_stage, "stc_cell_fwd_stage"))

    def region(name, k, width):
        o = lay[name] + k * R * width
        return saved[o:o + R * width].view(B, ne, C, width)

    def stage(which):
        _lib.check(run_stage(dims, which, Gc.data_ptr(), Xe.data_ptr(), ne * C * Din, He.data_ptr(), Wg.data_ptr(),
                             _ptr(bg), Wc.data_ptr(), _ptr(bc), Hn.data_ptr(), saved.data_ptr(), saved.numel() * 4,
                             stream), what)
        _lib.note_launches()

    def chain(term0, name, width, first):
        """Y_1 = Gs^T Y_0, Y_k = 2 Gs^T Y_{k-1} - Y_{k-2} into regions `name`[first ...]."""
        prev2, prev = None, term0
        for k in range(1, Ks):
            out = region(name, first + k - 1, width)
            if k == 1:
                ps.hop_ext(prev, out)
            else:
                ps.hop_ext(prev, out, Z_ext=prev2, alpha=2.0, beta=-1.0)
            prev2, prev = prev, out

    chain(Xe, "Yx", Din, 0)
    chain(He, "Yh", h, 0)
    stage(_lib.STAGE_GATES)
    chain(region("Yr", 0, h), "Yr", h, 1)
    stage(_lib.STAGE_CANDI)
    return Hn[:, :n].contiguous(), (Gc, Xe, He, Wg, Wc, saved), dims, lay


class _PartitionedCell(torch.autograd.Function):
    """One STC cell on this rank's node block; forward and backward are the C-ABI stages of include/stc_b200.h with
    the spatial hops (halo exchange + `stc_support_apply`) in between."""

    @staticmethod
    def forward(ctx, Gc, Xt, Ht_1, Wg, bg, Wc, bc, Ev, cfg):
        Hn, ctx.keep, ctx.dims, ctx.lay = _partitioned_forward(Gc, Xt, Ht_1, Wg, bg, Wc, bc, cfg, fwd_only=False)
        ctx.cfg = cfg
        ctx.has_bias = bg is not None
        # saved only so that autograd refuses a backward after an in-place change of the values
        ctx.save_for_backward(*([Ev] if Ev is not None else []))
        return Hn

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dHn):
        from . import _lib
        ps, Ks, Kc, activation, reduce_params = ctx.cfg
        Gc, Xe, He, Wg, Wc, saved = ctx.keep
        ctx.saved_tensors                        # raises if the edge values were changed in place since the forward
        dims = ctx.dims
        lib = _lib.load()
        B, ne, C, Din = Xe.shape
        h = He.shape[-1]
        n = ps.nloc
        dev = Xe.device
        stream = torch.cuda.current_stream().cuda_stream
        dHe = He.new_zeros(B, ne, C, h)          # halo rows carry no output gradient: they stay out of every dW
        dHe[:, :n] = dHn
        _lib.sync_deterministic()   # the scratch holds the partial slots of the fixed-order reductions while it is on
        scratch = torch.empty(lib.stc_cell_bwd_scratch_bytes(dims) // 4, dtype=torch.float32, device=dev)
        lay = _lib.scratch_layout(dims)
        R = B * ne * C
        dXe = torch.empty_like(Xe)
        dHp = torch.empty_like(He)
        P, L = Ks * Kc, Din + h
        need = ctx.needs_input_grad
        learn = need[7]                          # the edge values of a learnable support require grad
        # one flat buffer for every replicated-parameter gradient (and the [nnz] edge gradient): the all-reduce below
        # is a single call.  The ranks' edge-gradient slices are disjoint, so its sum is exact.
        sizes = [P * L * 2 * h, 2 * h if ctx.has_bias else 0, P * L * h, h if ctx.has_bias else 0, C * C,
                 ps.nnz if learn else 0]
        flat = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
        dWg, dbg, dWc, dbc, dGc, dEv = flat.split(sizes)
        pz = lambda t: t.data_ptr() if t.numel() else None

        def region(name, k, width, buf=scratch, offsets=lay):
            o = offsets[name] + k * R * width
            return buf[o:o + R * width].view(B, ne, C, width)

        fwd_term = lambda name, k, width: region(name, k, width, saved, ctx.lay)
        if learn:
            m = ps.maps()
            eg = lambda terms: dict(terms=terms, dvals=dEv[m.edge_lo:m.edge_hi])
        else:
            eg = lambda terms: {}

        def stage(which):
            _lib.check(lib.stc_cell_bwd_stage(dims, which, Gc.data_ptr(), Xe.data_ptr(), ne * C * Din, He.data_ptr(),
                                              Wg.data_ptr(), Wc.data_ptr(), dHe.data_ptr(), dXe.data_ptr(), dHp.data_ptr(),
                                              dWg.data_ptr(), pz(dbg), dWc.data_ptr(), pz(dbc), dGc.data_ptr(), 1,
                                              saved.data_ptr(), saved.numel() * 4, scratch.data_ptr(),
                                              scratch.numel() * 4, stream), "stc_cell_bwd_stage")
            _lib.note_launches()

        stage(_lib.STAGE_CANDI)
        dYr = [region("dYr", k, h) for k in range(Ks)]
        # A of each chain's hop k is the forward term Y_{k-1} the forward left in `saved` (Y_0: Xe, He, r*H)
        adjoint_chain_ext(ps, dYr, **eg([fwd_term("Yr", k, h) for k in range(Ks - 1)]))
        dYr[0][:, n:].zero_()                    # d(r*H) of the halo rows belongs to their owners
        stage(_lib.STAGE_GATES)
        adjoint_chain_ext(ps, [dXe] + [region("dYx", k, Din) for k in range(Ks - 1)],
                          **eg([Xe] + [fwd_term("Yx", k, Din) for k in range(Ks - 2)]))
        adjoint_chain_ext(ps, [dHp] + [region("dYh", k, h) for k in range(Ks - 1)],
                          **eg([He] + [fwd_term("Yh", k, h) for k in range(Ks - 2)]))
        if reduce_params and ps.world > 1:
            dist.all_reduce(flat, group=ps.group)
        return (dGc.view(C, C) if need[0] else None, dXe[:, :n].contiguous() if need[1] else None,
                dHp[:, :n].contiguous() if need[2] else None, dWg.view(P * L, 2 * h) if need[3] else None,
                dbg if (need[4] and ctx.has_bias) else None, dWc.view(P * L, h) if need[5] else None,
                dbc if (need[6] and ctx.has_bias) else None, dEv if learn else None, None)


def partitioned_cell_forward(ps: PartitionedSupport, Gc: torch.Tensor, Xt: torch.Tensor, Ht_1: torch.Tensor,
                             Wg: torch.Tensor, bg: Optional[torch.Tensor], Wc: torch.Tensor,
                             bc: Optional[torch.Tensor], Ks: int, Kc: int, activation=None,
                             reduce_params: bool = True) -> torch.Tensor:
    """`STC_Cell.forward` (`framework/STC_GNN.py:65-79`) on this rank's node block of a row-partitioned graph.

    Xt [B, nloc, C, Din], Ht_1 [B, nloc, C, h] are the local blocks; returns the local block of H'.  The spatial
    hops run here (halo exchange + `stc_support_apply`), the node-local stages are `stc_cell_fwd_stage` /
    `stc_cell_bwd_stage` (include/stc_b200.h).  Differentiable w.r.t. Gc, Xt, Ht_1, the parameters and, for a
    learnable support, its edge values `ps.vals` ([nnz], Gs-CSR order; the gradient is formed inside the adjoint hops
    and lands in this rank's slice of it).  The parameters, Gc and the edge values are replicated over the ranks, so
    their gradients are partial sums over this rank's nodes: with `reduce_params` (default) the backward all-reduces
    them in ONE flat bucket and every rank receives the full gradient (all ranks must then run the backward); pass
    False to reduce later, e.g. once per step through `dp.GradBucket` after a time loop (put the leaf behind the
    values -- `ps.vals`, or the raw parameter it is computed from -- into that bucket).
    """
    for name, t in (("Gc", Gc), ("Xt", Xt), ("Ht_1", Ht_1), ("gates.W", Wg), ("candi.W", Wc)):
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"partitioned cell: {name} must be a float32 CUDA tensor (there is no CPU path)")
    B, n, C, Din = Xt.shape
    h = Ht_1.shape[-1]
    if n != ps.nloc or Ht_1.shape != (B, n, C, h):
        raise RuntimeError(f"local block has {n} nodes, the partition owns {ps.nloc}; Ht_1 {tuple(Ht_1.shape)}")
    if (bg is None) != (bc is None):
        raise RuntimeError("partitioned cell: gates.b and candi.b must both be given or both be None")
    if B == 0:   # empty batch (the same on every rank: the batch is replicated, the nodes are split): nothing to exchange
        return Ht_1.new_zeros(0, n, C, h)
    cfg = (ps, Ks, Kc, activation, reduce_params)
    from .cell import forward_only
    if forward_only(Gc, Xt, Ht_1, Wg, bg, Wc, bc, ps.vals):   # no gradient can be asked for: no backward state
        return _partitioned_forward(Gc, Xt, Ht_1, Wg, bg, Wc, bc, cfg, fwd_only=True)[0]
    return _PartitionedCell.apply(Gc, Xt, Ht_1, Wg, bg, Wc, bc, ps.vals, cfg)
