"""Recurrent roll-out that drives the cell: the reference's STC_Encoder (layers x T) followed by the
STC_Decoder horizon loop (/root/reference/framework/STC_GNN.py:97-123, 154-166, 194-204) with the
supports handed in -- i.e. STCGNN.forward minus MGP_Gen and out_proj.  This is the unit bench.py times
("one sample = one [T,N,C] window through all layers and timesteps") and the only way to drive
configurations whose N makes the reference's MixedFusion (N^2 x N^2 weights) unconstructible.
"""
from __future__ import annotations

import torch
from torch import nn

from . import _lib
from .cell import STC_Cell, _csr_cache
from .support import CsrSupport, dense_struct, support_apply


class _XSideTerms(torch.autograd.Function):
    """Spatial terms of the WHOLE input sequence in one launch (SURVEY 8f row f1; Ks = 2, dense Gs).

    In the encoder's first layer Xt does not depend on the recurrence (`framework/STC_GNN.py:107-118`), and with the
    shipped input width (Din = 1, C = 5) a per-step product is 5 floats wide: it runs on the general FFMA kernels at
    0.05 of HBM bandwidth, 18 + 9 launches per step.  Here the sequence is regrouped as [B, N, T*C*Din] (padded to a
    multiple of 4 columns) so that ONE tensor-core `stc_support_apply` produces Y_1 = Gs^T X for all T, and the backward
    folds all T adjoints into dGs with ONE `stc_support_outer`.  Outputs: T tensors [1, B, N, C, Din] (= [Ks-1, ...]),
    handed to the cells as `_Yx`.  The input sequence itself gets no gradient through this path (callers hoist only
    when it needs none)."""

    @staticmethod
    def forward(ctx, Gs, X_seq):
        B, T, N, C, Din = X_seq.shape
        W = T * C * Din
        Wp = (W + 3) & ~3
        Xp = X_seq.new_zeros(B, N, Wp) if Wp != W else X_seq.new_empty(B, N, Wp)
        Xp[:, :, :W] = X_seq.permute(0, 2, 1, 3, 4).reshape(B, N, W)
        Gs_c = Gs.detach().contiguous()
        Y1p = support_apply(Gs_c, Xp, transpose=True)
        outs = tuple(Y1p[:, :, t * C * Din:(t + 1) * C * Din].reshape(1, B, N, C, Din).contiguous() for t in range(T))
        ctx.save_for_backward(Gs_c, Xp)
        ctx.shape = (B, T, N, C, Din, W, Wp)
        return outs

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *dY):
        Gs, Xp = ctx.saved_tensors
        B, T, N, C, Din, W, Wp = ctx.shape
        if not ctx.needs_input_grad[0]:
            return None, None
        dYp = Xp.new_zeros(B, N, Wp) if Wp != W else Xp.new_empty(B, N, Wp)
        for t, g in enumerate(dY):
            piece = dYp[:, :, t * C * Din:(t + 1) * C * Din]
            if g is None:
                piece.zero_()
            else:
                piece.copy_(g.reshape(B, N, C * Din))
        dGs = torch.zeros(N, N, dtype=torch.float32, device=Xp.device)
        lib = _lib.load()
        _lib.check(lib.stc_support_outer(N, B, Wp, Xp.data_ptr(), N * Wp, dYp.data_ptr(), 1.0, dGs.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream), "stc_support_outer")
        _lib.note_launches()
        return dGs, None


def _hoistable(Gs, X_seq: torch.Tensor, cell: STC_Cell) -> bool:
    """One batched launch pays when the per-step product is narrow (the shipped Din = 1) and nothing needs dX_seq."""
    if not isinstance(Gs, torch.Tensor) or Gs.layout != torch.strided or not Gs.is_cuda or Gs.dtype != torch.float32:
        return False
    B, T, N, C, Din = X_seq.shape
    narrow = (C * Din) % 4 != 0 or C * Din < 32
    return (cell.Ks == 2 and narrow and T >= 2 and B > 0 and N <= 128 and not X_seq.requires_grad and X_seq.is_cuda
            and X_seq.dtype == torch.float32)


def share_plan(layers: int, T: int, horizon: int) -> dict:
    """Which cell computes the spatial terms of each hidden state that two cells read, and which cell takes them.

    Cells are ("enc", layer, t) and ("dec", layer, step); a side is "x" (the cell reads the state as Xt) or "h" (as
    Ht_1).  Every hidden state of the roll-out is read by at most two cells, and both hop it the same way (same Gs, same
    width C*h), so the terms are computed once: by the reader that runs first in forward (the encoder is layer-major),
    and handed to the other.  Returns
      pairs  [((producer cell, side), (consumer cell, side)), ...] in the producer's forward order;
      zero   [(cell, "h"), ...]: the encoder's zero initial states, whose terms are exactly 0 (no hop, no chain).
    A state that one cell reads on both sides (the decoder of a one-layer stack) is not shared."""
    order, readers = [], {}

    def read(cell, side, state):
        if state is not None:
            readers.setdefault(state, []).append((cell, side))

    for l in range(layers):
        for t in range(T):
            cell = ("enc", l, t)
            order.append(cell)
            read(cell, "x", None if l == 0 else ("enc", l - 1, t))     # layer 0 reads the input sequence
            read(cell, "h", None if t == 0 else ("enc", l, t - 1))
    for s in range(horizon):
        x = ("enc", layers - 1, T - 1) if s == 0 else ("dec", layers - 1, s - 1)
        for l in range(layers):
            cell = ("dec", l, s)
            order.append(cell)
            read(cell, "x", x if l == 0 else ("dec", l - 1, s))
            read(cell, "h", ("enc", l, T - 1) if s == 0 else ("dec", l, s - 1))
    rank = {c: i for i, c in enumerate(order)}
    pairs = []
    for rs in readers.values():
        if len(rs) == 2 and rs[0][0] != rs[1][0]:
            first, second = sorted(rs, key=lambda r: rank[r[0]])
            pairs.append((first, second))
    pairs.sort(key=lambda pr: rank[pr[0][0]])
    zero = [(("enc", l, 0), "h") for l in range(layers)] if T > 0 else []
    return {"pairs": pairs, "zero": zero}


def _shares_terms(Gs, cell: STC_Cell) -> bool:
    """Shared terms need one support every cell hops the same way: a dense fp32 CUDA tensor or a CsrSupport (a row-
    partitioned support keeps its own exchange path), and at least one spatial term."""
    if cell.Ks < 2:
        return False
    if isinstance(Gs, CsrSupport):
        return True
    return isinstance(Gs, torch.Tensor) and Gs.layout == torch.strided and Gs.is_cuda and Gs.dtype == torch.float32


class RecurrentStack(nn.Module):
    def __init__(self, num_nodes: int, num_categories: int, Ks: int, Kc: int, input_dim: int, hidden_dim: int,
                 num_layers: int, out_horizon: int, use_bias=True, activation=None):
        super().__init__()
        self.num_layers, self.out_horizon, self.hidden_dim = num_layers, out_horizon, hidden_dim
        # construction order = the reference's (encoder cells, then decoder cells) for seeded-init parity
        self.encoder = nn.ModuleList(
            STC_Cell(num_nodes, num_categories, Ks, Kc, input_dim if i == 0 else hidden_dim, hidden_dim,
                     use_bias=use_bias, activation=activation) for i in range(num_layers))
        self.decoder = nn.ModuleList(
            STC_Cell(num_nodes, num_categories, Ks, Kc, hidden_dim, hidden_dim, use_bias=use_bias,
                     activation=activation) for _ in range(num_layers))

    def forward(self, Gs, Gc: torch.Tensor, X_seq: torch.Tensor) -> torch.Tensor:
        """X_seq [B,T,N,C,Din] -> decoder hidden states [B,horizon,N,C,h] (out_horizon = 0: the last encoder
        layer's hidden states [B,T,N,C,h])."""
        assert X_seq.dim() == 5, "X_seq must be [B,T,N,C,Din]"
        B, T = X_seq.shape[0], X_seq.shape[1]
        if isinstance(Gs, torch.Tensor) and Gs.layout != torch.strided:
            Gs = _csr_cache(Gs)    # one CsrSupport for every cell (what each cell would look up itself)
        step = self._shared_steps(Gs, Gc, T)
        # Layer l > 0 consumes layer l-1's per-step outputs directly: the reference stacks them and slices the stack
        # again (STC_GNN.py:114,111), which in backward costs one zero-filled [B,T,N,C,h] tensor plus one full-size
        # add per timestep (select_backward) -- same values, none of that traffic.
        seq = [X_seq[:, t] for t in range(T)]
        last = []
        for li, cell in enumerate(self.encoder):
            Ht = cell.init_hidden(B)
            outs = []
            # layer 0: the Xt-side spatial terms of all T steps from one batched launch (row f1)
            yx = _XSideTerms.apply(Gs, X_seq) if (li == 0 and _hoistable(Gs, X_seq, cell)) else None
            for t in range(T):
                yx_t = None if yx is None else yx[t]
                if step is None:
                    Ht = cell(Gs=Gs, Gc=Gc, Xt=seq[t], Ht_1=Ht, _Yx=yx_t)
                else:
                    Ht = step(cell, ("enc", li, t), seq[t], Ht, yx_t)
                outs.append(Ht)
            seq = outs
            last.append(Ht)
        if self.out_horizon == 0:   # encoder only (the large synthetic graphs drive STC_Encoder directly, SURVEY 8d)
            return torch.stack(seq, dim=1)
        states, x, outs = last, last[-1], []
        for _ in range(self.out_horizon):
            new_states, inp = [], x
            for l, cell in enumerate(self.decoder):
                if step is None:
                    inp = cell(Gs=Gs, Gc=Gc, Xt=inp, Ht_1=states[l])
                else:
                    inp = step(cell, ("dec", l, len(outs)), inp, states[l], None)
                new_states.append(inp)
            states, x = new_states, new_states[-1]
            outs.append(x)
        return torch.stack(outs, dim=1)

    def _shared_steps(self, Gs, Gc, T: int):
        """The cell step of forward() with the terms of share_plan handed from producer to consumer, or None when the
        support or the cells do not qualify (_shares_terms; a row-partitioned support keeps its own exchange path)."""
        cells = list(self.encoder) + list(self.decoder)
        if not cells or not all(_shares_terms(Gs, c) for c in cells) or len({c.Ks for c in cells}) != 1:
            return None
        plan = share_plan(self.num_layers, T, self.out_horizon)
        give = {}
        for pc, pside in sorted((p for p, _ in plan["pairs"]), key=lambda p: p[1]):   # "h" after "x"
            give[pc] = give.get(pc, ()) + (pside,)
        take = {}
        for producer, (cc, cside) in plan["pairs"]:
            take.setdefault(cc, {})[cside] = producer
        zero = {c for c, _ in plan["zero"]}
        given = {}            # (producer cell, side) -> its terms, until the consumer has taken them
        Ks = cells[0].Ks

        def step(cell, key, Xt, H, yx):
            src = take.get(key, {})
            yx_shared = "x" in src
            if yx_shared:
                yx = given.pop(src["x"])
            yh = given.pop(src["h"]) if "h" in src else None
            if key in zero:   # the zero initial state: its terms are zeros too (Ks = 2: the state itself)
                yh = H.unsqueeze(0) if Ks == 2 else H.new_zeros((Ks - 1,) + tuple(H.shape))
            g = give.get(key, ())
            out = cell._shared_step(Gs, Gc, Xt, H, yx, yh, g, yx_shared)
            if not g:
                return out
            for side, terms in zip(g, out[1:]):
                given[(key, side)] = terms
            return out[0]

        return step
