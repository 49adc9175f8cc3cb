"""Drop-in replacement for the reference's STC_Cell (/root/reference/framework/STC_GNN.py:51-79).

Same constructor, ``forward(Gs, Gc, Xt, Ht_1)``, ``init_hidden`` and parameter names
(``gates.W``, ``gates.b``, ``candi.W``, ``candi.b``) so ``load_state_dict(strict=True)`` of a reference
checkpoint works and a seeded construction draws the same weights; the internals are one call into
libstc_b200.so per direction (include/stc_b200.h).  CUDA fp32 only -- anything else raises.
"""
from __future__ import annotations

import os
from types import SimpleNamespace

import torch
from torch import nn

from . import _lib
from .support import CsrSupport, dense_struct

# Gradients of LEAF tensors (the cell's parameters; Gs / Gc when they are leaves) are accumulated by the backward
# kernels straight into `.grad` (the ABI's accumulate mode) instead of being returned to autograd: a cell is applied
# T times per sequence and the supports feed all 24 cell steps, so the returned form costs one freshly zeroed buffer
# set (6 memsets) per cell backward plus one elementwise add per tensor and step (~250 tiny launches per SF step,
# profiles/r1q_launches.txt).  Semantics are those of `loss.backward()` (gradients add into `.grad`);
# `torch.autograd.grad(...)` w.r.t. these leaves needs the returned form: set STC_INPLACE_GRADS=0 or
# `stc_gnn_b200.cell.INPLACE_LEAF_GRADS = False`.
INPLACE_LEAF_GRADS = os.environ.get("STC_INPLACE_GRADS", "1") != "0"

# A cell call that no gradient can be asked of (torch.no_grad / torch.inference_mode, or no tensor input requires grad)
# runs the forward-only form (stc_cell_fwd_only): no autograd node, a workspace without the regions only the backward
# reads (r, c, the P_1 partials), and bitwise the same output.  STC_FORWARD_ONLY=0 or
# `stc_gnn_b200.cell.FORWARD_ONLY = False` keeps the training forward for such calls too (A/B runs).
FORWARD_ONLY = os.environ.get("STC_FORWARD_ONLY", "1") != "0"

_ACT_CODES = {None: _lib.ACT_NONE, nn.ReLU: _lib.ACT_RELU}
_ACT_NAMES = {_lib.ACT_NONE: None, _lib.ACT_RELU: "relu"}


def _activation_code(activation) -> int:
    if activation in _ACT_CODES:
        return _ACT_CODES[activation]
    if isinstance(activation, str):
        return {"none": _lib.ACT_NONE, "relu": _lib.ACT_RELU}[activation]
    raise NotImplementedError(f"activation {activation!r} is not implemented in the B200 cell (None or nn.ReLU)")


class GraphConvParams(nn.Module):
    """Parameter holder with the reference BDG_Dif's names, shapes and init (STC_GNN.py:16-22):
    W [(input_dim*Ks*Kc), hidden_dim] xavier-normal, b [hidden_dim] zeros."""

    def __init__(self, Ks: int, Kc: int, input_dim: int, hidden_dim: int, use_bias: bool = True):
        super().__init__()
        self.Ks, self.Kc, self.input_dim, self.hidden_dim, self.use_bias = Ks, Kc, input_dim, hidden_dim, use_bias
        self.W = nn.Parameter(torch.empty(input_dim * Ks * Kc, hidden_dim), requires_grad=True)
        nn.init.xavier_normal_(self.W)
        if use_bias:
            self.b = nn.Parameter(torch.empty(hidden_dim), requires_grad=True)
            nn.init.constant_(self.b, val=0.0)


def _dims(B, N, C, Din, h, Ks, Kc, act, has_bias) -> _lib.StcDims:
    return _lib.StcDims(B, N, C, Din, h, Ks, Kc, act, 1 if has_bias else 0)


_SIZES = {}


def _buffer_floats(lib, dims: _lib.StcDims, key):
    """(saved, scratch) buffer sizes in floats of a cell call, cached per shape and deterministic mode (the scratch holds
    the partial slots while it is on): at the reference's batch size a training step is bound by host-side call
    overhead (48 cell calls), so the two size queries are not repeated."""
    key = key + (_lib.sync_deterministic(),)
    hit = _SIZES.get(key)
    if hit is None:
        if len(_SIZES) > 256:
            _SIZES.clear()
        hit = _SIZES[key] = (lib.stc_cell_saved_bytes(dims) // 4, lib.stc_cell_bwd_scratch_bytes(dims) // 4)
    return hit


def _fwd_only_floats(lib, dims: _lib.StcDims, key):
    """Workspace size in floats of a forward-only cell call, cached per shape like _buffer_floats."""
    key = ("fwd_only",) + key
    hit = _SIZES.get(key)
    if hit is None:
        if len(_SIZES) > 256:
            _SIZES.clear()
        hit = _SIZES[key] = lib.stc_cell_fwd_only_bytes(dims) // 4
    return hit


def forward_only(*tensors) -> bool:
    """True when a cell call over these tensor inputs takes the forward-only form: FORWARD_ONLY is on and autograd
    cannot ask for a gradient (grad mode off, which includes inference mode, or no input requires grad)."""
    return FORWARD_ONLY and not (torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors))


def _ptr(t):
    return t.data_ptr() if t is not None else None


_SAVED_OFFSETS = {}


def _terms_view(saved, dims, key, side, shape, fwd_only=False):
    """The spatial terms [Ks-1,B,N,C,w] a cell call computed for one side: a view of its `saved` buffer (of its
    forward-only workspace with `fwd_only`)."""
    offs = _SAVED_OFFSETS.get((key, fwd_only))
    if offs is None:
        if len(_SAVED_OFFSETS) > 256:
            _SAVED_OFFSETS.clear()
        offs = _SAVED_OFFSETS[(key, fwd_only)] = _lib.saved_layout(dims, fwd_only)
    n = 1
    for s_ in shape:
        n *= s_
    return saved[offs["Yx" if side == "x" else "Yh"]:][:n].view(shape)


def _run_forward(Gs, Gc, Xt, H, Wg, bg, Wc, bc, Yx, Ev, cfg, Yh, give, fwd_only):
    """Argument checks and the forward launch of one cell step, shared by the training form (_CellFunction, which
    fills `saved` for its backward) and the forward-only form (fwd_only: stc_cell_fwd_only on the smaller workspace).
    Inputs as in _CellFunction; `give` the sides whose computed terms are returned.  Returns the contiguous operands the
    launch read, the buffer it filled (`buf`), H' (`Hn`) and the given terms (`given`, views of `buf`)."""
    lib = _lib.load()
    Ks, Kc, act = cfg
    B, N, C, Din = Xt.shape
    h = H.shape[-1]
    for name, t in (("Gc", Gc), ("Xt", Xt), ("Ht_1", H), ("gates.W", Wg), ("candi.W", Wc)):
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError(f"STC_Cell (B200): {name} must be a float32 CUDA tensor, got {t.dtype} on {t.device}; "
                               "there is no CPU fallback")
    if H.shape != (B, N, C, h):
        raise RuntimeError(f"Ht_1 shape {tuple(H.shape)} does not match Xt {tuple(Xt.shape)}")
    rows = (Din + h) * Ks * Kc
    if Wg.shape != (rows, 2 * h) or Wc.shape != (rows, h) or Gc.shape != (C, C):
        raise RuntimeError(f"shape mismatch: gates.W {tuple(Wg.shape)} (want {(rows, 2 * h)}), candi.W "
                           f"{tuple(Wc.shape)} (want {(rows, h)}), Gc {tuple(Gc.shape)} (want {(C, C)})")
    for name, b_, n_ in (("gates.b", bg, 2 * h), ("candi.b", bc, h)):
        if b_ is not None and (b_.shape != (n_,) or not b_.is_cuda or b_.dtype != torch.float32):
            raise RuntimeError(f"{name} must be a float32 CUDA tensor of shape ({n_},)")
    if (bg is None) != (bc is None):
        raise RuntimeError("gates.b and candi.b must both be present or both absent")
    csr = isinstance(Gs, CsrSupport)
    gs_keep = None
    if csr:
        if Gs.N != N:
            raise RuntimeError(f"CSR support has {Gs.N} nodes, Xt has {N}")
        if Gs.batch is not None and Gs.batch != B:
            raise RuntimeError(f"per-sample CSR support has values for B = {Gs.batch} samples, Xt has B = {B}")
        if Ev is not None and Ev is not Gs.vals:
            raise RuntimeError("edge values passed to the cell must be the CsrSupport's own `vals`")
        if Gs.learnable or Gs.batch is not None:   # the values may have changed since the last step (optimizer update,
            Gs.sync_t_vals()                       # new with_values, an in-place write)
        gs_struct = Gs.struct()
    else:
        if not Gs.is_cuda or Gs.dtype != torch.float32 or Gs.shape != (N, N):
            raise RuntimeError(f"Gs must be a float32 CUDA [N,N] tensor or a CsrSupport, got {tuple(Gs.shape)} {Gs.dtype}")
        gs_keep = Gs.contiguous()
        gs_struct = dense_struct(gs_keep)
    Gc_c, H_c, Wg_c, Wc_c = Gc.contiguous(), H.contiguous(), Wg.contiguous(), Wc.contiguous()
    bg_c = bg.contiguous() if bg is not None else None
    bc_c = bc.contiguous() if bc is not None else None
    # the encoder's [:, t] view keeps each sample's [N,C,Din] slab contiguous: pass the batch stride
    Xt_c = Xt if (B == 0 or Xt[0].is_contiguous()) else Xt.contiguous()
    xbs = Xt_c.stride(0) if B > 1 else N * C * Din
    dims = _dims(B, N, C, Din, h, Ks, Kc, act, bg is not None)
    size_key = (B, N, C, Din, h, Ks, Kc, act, bg is not None)
    floats = _fwd_only_floats(lib, dims, size_key) if fwd_only else _buffer_floats(lib, dims, size_key)[0]
    buf = torch.empty(floats, dtype=torch.float32, device=Xt.device)
    Hn = torch.empty((B, N, C, h), dtype=torch.float32, device=Xt.device)
    stream = torch.cuda.current_stream().cuda_stream

    def supplied(Y, w, what):
        if Y is None or Ks <= 1:
            return None
        if Y.shape != (Ks - 1, B, N, C, w) or not Y.is_cuda or Y.dtype != torch.float32:
            raise RuntimeError(f"supplied {what} terms must be a float32 CUDA tensor of shape {(Ks - 1, B, N, C, w)}, "
                               f"got {tuple(Y.shape)}")
        return Y.contiguous()

    Yx_c, Yh_c = supplied(Yx, Din, "Xt-side"), supplied(Yh, h, "H-side")
    for side in give:
        if side not in ("x", "h") or Ks <= 1 or (Yx_c if side == "x" else Yh_c) is not None:
            raise RuntimeError(f"a cell can only give terms of a side it computes itself (give={give!r}, Ks={Ks})")
    args = (dims, gs_struct, Gc_c.data_ptr(), Xt_c.data_ptr(), xbs, H_c.data_ptr(), Wg_c.data_ptr(), _ptr(bg_c),
            Wc_c.data_ptr(), _ptr(bc_c), Hn.data_ptr(), buf.data_ptr(), buf.numel() * 4)
    if B == 0:
        status = 0
    elif fwd_only:
        status = lib.stc_cell_fwd_only(*args, _ptr(Yx_c), _ptr(Yh_c), stream)
    elif Yx_c is not None or Yh_c is not None:
        status = lib.stc_cell_fwd_x(*args, _ptr(Yx_c), _ptr(Yh_c), stream)
    else:
        status = lib.stc_cell_fwd(*args, stream)
    _lib.check(status, "stc_cell_fwd_only" if fwd_only else "stc_cell_fwd")
    _lib.note_launches()
    given = tuple(_terms_view(buf, dims, size_key, side, (Ks - 1, B, N, C, Din if side == "x" else h), fwd_only)
                  for side in give)
    return SimpleNamespace(Hn=Hn, buf=buf, given=given, Gs=gs_keep, Gc=Gc_c, Xt=Xt_c, H=H_c, Wg=Wg_c, Wc=Wc_c, Yx=Yx_c,
                           Yh=Yh_c, xbs=xbs, csr=csr, size_key=size_key, dims_tuple=(B, N, C, Din, h))


class _CellFunction(torch.autograd.Function):
    """One cell step. Inputs that may need gradients: Gs (dense only), Gc, Xt, H, Wg, bg, Wc, bc, `Ev`, the edge values
    [nnz] of a learnable CsrSupport Gs (the support object itself is not a tensor autograd can see; Ev is its `vals`),
    and caller-supplied spatial terms of either side (stack.py): `Yx` [Ks-1,B,N,C,Din] of Xt and `Yh` [Ks-1,B,N,C,h] of
    H.  No hop runs for a supplied side, and the gradient of its terms is returned un-folded.

    `share` = (give, yx_shared):
      give       sides ("x", "h") whose computed terms are also returned (views of `saved`), after H' in that order; the
                 gradient arriving at them (from the cell that took them) is folded in before this cell's own adjoint
                 chain of that side, so one hop and one dGs product serve both readers.
      yx_shared  the supplied `Yx` came from another cell that folds their adjoint into the chain of Xt itself: then
                 Xt's own gradient is its direct term only.  Without it (the _XSideTerms path, which folds only into
                 dGs) Xt may not need a gradient."""

    @staticmethod
    def forward(ctx, Gs, Gc, Xt, H, Wg, bg, Wc, bc, Yx, Ev, cfg, Yh=None, share=None):
        give, yx_shared = share if share is not None else ((), False)
        f = _run_forward(Gs, Gc, Xt, H, Wg, bg, Wc, bc, Yx, Ev, cfg, Yh, give, fwd_only=False)
        ctx.size_key = f.size_key
        ctx.hoisted, ctx.h_given, ctx.yx_shared, ctx.give = f.Yx is not None, f.Yh is not None, bool(yx_shared), tuple(give)
        ctx.cfg, ctx.dims_tuple, ctx.xbs, ctx.csr = cfg, f.dims_tuple, f.xbs, f.csr
        ctx.gs_obj = Gs if f.csr else None
        ctx.has_bias = bg is not None
        # leaves whose gradient the backward adds into `.grad` directly (index = position among forward's inputs)
        ctx.sinks = {}
        if INPLACE_LEAF_GRADS:
            for i, t in ((0, None if f.csr else Gs), (1, Gc), (4, Wg), (5, bg), (6, Wc), (7, bc), (9, Ev)):
                if t is not None and ctx.needs_input_grad[i] and t.is_leaf and t.is_contiguous():
                    ctx.sinks[i] = t
        ctx.has_ev = Ev is not None
        ctx.save_for_backward(*( [] if f.csr else [f.Gs] ), f.Gc, f.Xt, f.H, f.Wg, f.Wc, f.buf,
                              *([f.Yx] if f.Yx is not None else []), *([f.Yh] if f.Yh is not None else []),
                              *([Ev] if Ev is not None else []))
        if not give:
            return f.Hn
        ctx.set_materialize_grads(False)   # no gradient for given terms: nothing to fold (rather than a zero tensor)
        return (f.Hn,) + f.given

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dHn, *dGiven):
        lib = _lib.load()
        Ks, Kc, act = ctx.cfg
        B, N, C, Din, h = ctx.dims_tuple
        sv = list(ctx.saved_tensors)
        if ctx.has_ev:
            sv.pop()   # saved only so that autograd refuses a backward after an in-place change of the values
        Yh = sv.pop() if ctx.h_given else None
        Yx = sv.pop() if ctx.hoisted else None
        if ctx.csr:
            Gs = ctx.gs_obj
            Gc, Xt, H, Wg, Wc, saved = sv
            gs_struct = Gs.struct()
        else:
            Gs, Gc, Xt, H, Wg, Wc, saved = sv
            gs_struct = dense_struct(Gs)
        n_in = len(ctx.needs_input_grad)   # Yh and share are optional trailing inputs
        need = tuple(ctx.needs_input_grad) + (False,) * (13 - n_in)  # Gs, Gc, Xt, H, Wg, bg, Wc, bc, Yx, Ev, cfg, Yh, share
        dev = H.device
        dHn = dHn.contiguous() if dHn is not None else torch.zeros(B, N, C, h, dtype=torch.float32, device=dev)
        L, P = Din + h, Ks * Kc
        dims = _dims(B, N, C, Din, h, Ks, Kc, act, ctx.has_bias)
        new = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
        if ctx.hoisted and need[2] and not ctx.yx_shared:
            raise RuntimeError("hoisted Xt-side terms: the gradient w.r.t. Xt is folded by the caller (stack.py hoists only "
                               "when the input sequence needs no gradient)")
        dXt = new(B, N, C, Din) if need[2] else None
        dH = new(B, N, C, h)
        dYx = torch.empty_like(Yx) if ctx.hoisted and need[8] else None
        dYh = torch.empty_like(Yh) if ctx.h_given and need[11] else None
        fold = {side: g.contiguous() for side, g in zip(ctx.give, dGiven) if g is not None and B > 0}
        returned = [None] * 13

        def target(i, shape, wanted=True):
            """Buffer the kernels ADD input i's gradient into: the leaf's own `.grad` (created zeroed on first use in a
            step; nothing is returned to autograd), else a fresh zeroed tensor that is returned."""
            if not wanted:
                return None
            leaf = ctx.sinks.get(i)
            if leaf is not None and need[i]:
                if leaf.grad is None:
                    leaf.grad = torch.zeros(shape, dtype=torch.float32, device=dev)
                if leaf.grad.is_contiguous() and leaf.grad.dtype == torch.float32 and leaf.grad.shape == torch.Size(shape):
                    return leaf.grad
            buf = torch.zeros(shape, dtype=torch.float32, device=dev)
            returned[i] = buf
            return buf

        dWg, dWc = target(4, (P * L, 2 * h)), target(6, (P * L, h))
        dbg, dbc = target(5, (2 * h,), ctx.has_bias), target(7, (h,), ctx.has_bias)
        # a CSR support's gradient is that of its edge values: [nnz] in Gs-CSR order ([B, nnz] per sample)
        dGs = target(9, tuple(Gs.vals.shape), need[9]) if ctx.csr else target(0, (N, N), need[0])
        dGc = target(1, (C, C), need[1])
        returned[2], returned[3], returned[8], returned[11] = dXt, dH, dYx, dYh
        if B == 0:  # empty batch: every parameter gradient is zero (the targets are zeroed or untouched), nothing to launch
            for t in (dYx, dYh):
                if t is not None:
                    t.zero_()
            return tuple(returned[:n_in])
        scratch = torch.empty(_buffer_floats(lib, dims, ctx.size_key)[1], dtype=torch.float32, device=dev)
        common = (dims, gs_struct, Gc.data_ptr(), Xt.data_ptr(), ctx.xbs, H.data_ptr(), Wg.data_ptr(),
                  Wc.data_ptr(), dHn.data_ptr(), _ptr(dXt), dH.data_ptr(), dWg.data_ptr(), _ptr(dbg),
                  dWc.data_ptr(), _ptr(dbc), _ptr(dGs), _ptr(dGc), 1, saved.data_ptr(),
                  saved.numel() * 4, scratch.data_ptr(), scratch.numel() * 4)
        stream = torch.cuda.current_stream().cuda_stream
        if ctx.hoisted or ctx.h_given or fold:
            fx, fh = fold.get("x"), fold.get("h")
            status = lib.stc_cell_bwd_x(*common, _ptr(Yx), _ptr(dYx), _ptr(fx), _ptr(Yh), _ptr(dYh), _ptr(fh), stream)
        else:
            status = lib.stc_cell_bwd(*common, stream)
        _lib.check(status, "stc_cell_bwd")
        _lib.note_launches()
        for i in (0, 1, 4, 5, 6, 7, 8, 9, 11):    # inputs that need no gradient get none, whatever was computed for them
            if not need[i]:
                returned[i] = None
        return tuple(returned[:n_in])


def _cell(Gs, Gc, Xt, H, Wg, bg, Wc, bc, Yx, Ev, cfg, Yh=None, share=None):
    """One cell step (inputs as in _CellFunction): the training form when autograd may ask for a gradient, else the
    forward-only form (see FORWARD_ONLY), which returns the same values without an autograd node."""
    if not forward_only(Gs if isinstance(Gs, torch.Tensor) else None, Gc, Xt, H, Wg, bg, Wc, bc, Yx, Ev, Yh):
        extra = () if Yh is None and share is None else (Yh, share)
        return _CellFunction.apply(Gs, Gc, Xt, H, Wg, bg, Wc, bc, Yx, Ev, cfg, *extra)
    give = share[0] if share is not None else ()
    f = _run_forward(Gs, Gc, Xt, H, Wg, bg, Wc, bc, Yx, Ev, cfg, Yh, give, fwd_only=True)
    return (f.Hn,) + f.given if give else f.Hn


def stc_cell_forward(Gs, Gc, Xt, Ht_1, Wg, bg, Wc, bc, Ks: int, Kc: int, activation=None) -> torch.Tensor:
    """Functional form of the cell: H' = STC_Cell(Gs, Gc, Xt, Ht_1) with explicit weights (differentiable)."""
    return _cell(Gs, Gc, Xt, Ht_1, Wg, bg, Wc, bc, None, _edge_values(Gs), (int(Ks), int(Kc), _activation_code(activation)))


def _edge_values(Gs):
    """The edge values of a learnable CsrSupport (a tensor input of the cell, so autograd routes their gradient)."""
    return Gs.vals if isinstance(Gs, CsrSupport) and Gs.learnable else None


class STC_Cell(nn.Module):
    """B200 cell with the reference's public surface (STC_GNN.py:51-79).

    Deliberately NOT a subclass of the reference class: the reference's ``super(STC_Cell, self).__init__()``
    resolves the name through its module globals, which ``install()`` rebinds to this class.
    """

    def __init__(self, num_nodes: int, num_categories: int, Ks: int, Kc: int, input_dim: int, hidden_dim: int,
                 use_bias=True, activation=None):
        super().__init__()
        self.num_nodes = num_nodes
        self.num_categories = num_categories
        self.hidden_dim = hidden_dim
        self.input_dim = input_dim
        self.Ks, self.Kc = Ks, Kc
        self._act = _activation_code(activation)
        # same construction order as the reference (gates first) so seeded init reproduces its weights
        self.gates = GraphConvParams(Ks, Kc, input_dim + hidden_dim, hidden_dim * 2, use_bias)
        self.candi = GraphConvParams(Ks, Kc, input_dim + hidden_dim, hidden_dim, use_bias)

    def init_hidden(self, batch_size: int):
        weight = next(self.parameters()).data
        return weight.new_zeros(batch_size, self.num_nodes, self.num_categories, self.hidden_dim)

    def _shared_step(self, Gs, Gc, Xt, Ht_1, Yx=None, Yh=None, give=(), yx_shared=False):
        """One step of RecurrentStack with spatial terms shared between the two cells that read a hidden state
        (dense or CSR Gs): see _CellFunction.  Returns H' or, with `give`, (H', the terms of each side given)."""
        return _cell(Gs, Gc, Xt, Ht_1, self.gates.W, getattr(self.gates, "b", None), self.candi.W,
                     getattr(self.candi, "b", None), Yx, _edge_values(Gs), (self.Ks, self.Kc, self._act), Yh,
                     (give, yx_shared))

    def forward(self, Gs, Gc: torch.Tensor, Xt: torch.Tensor, Ht_1: torch.Tensor, _Yx: torch.Tensor = None):
        """`_Yx` (not part of the reference's signature): the spatial terms of Xt, [Ks-1,B,N,C,Din], when the caller
        produced them for a whole sequence at once (stack.py); their gradient comes back un-folded."""
        assert len(Xt.shape) == len(Ht_1.shape) == 4, 'STC-cell must take in 4D tensor as input [Xt, Ht-1]'
        if isinstance(Gs, torch.Tensor) and Gs.layout != torch.strided:
            Gs = _csr_cache(Gs)
        if hasattr(Gs, "fwd") and hasattr(Gs, "hop_ext"):
            # a halo.PartitionedSupport: Xt / Ht_1 are this rank's node blocks (construct the cell with num_nodes = the
            # local count so that init_hidden matches); spatial hops exchange halos, everything else is node-local
            from .halo import partitioned_cell_forward
            return partitioned_cell_forward(Gs, Gc, Xt, Ht_1, self.gates.W, getattr(self.gates, "b", None), self.candi.W,
                                            getattr(self.candi, "b", None), self.Ks, self.Kc, _ACT_NAMES[self._act],
                                            reduce_params=getattr(Gs, "reduce_per_cell", True))
        return _cell(Gs, Gc, Xt, Ht_1, self.gates.W, getattr(self.gates, "b", None), self.candi.W,
                     getattr(self.candi, "b", None), _Yx, _edge_values(Gs), (self.Ks, self.Kc, self._act))


_CSR_CACHE = {}


def _csr_cache(G: torch.Tensor) -> CsrSupport:
    """torch sparse tensors are converted once per (storage, version, structure) -- building Gs^T is not free.

    The entry keeps the keyed tensor alive: while it is cached its buffers cannot be freed and handed to a
    different sparse tensor at the same address, so a hit always means "this very tensor, unmodified"."""
    if G.requires_grad:
        raise RuntimeError("STC_Cell (B200): a torch sparse Gs is a constant support and gets no gradient; for learned "
                           "edge weights on a fixed pattern pass CsrSupport(rowptr, col, vals_requiring_grad, N) "
                           "(or a dense [N,N] tensor when the whole dGs is needed)")
    if G.layout == torch.sparse_csr:
        vals, idx = G.values(), G.col_indices()
    else:
        vals, idx = G._values(), G._indices()
    key = (vals.data_ptr(), vals._version, idx.data_ptr(), idx._version, int(vals.numel()), tuple(G.shape), G.layout,
           vals.dtype)
    hit = _CSR_CACHE.get(key)
    if hit is None:
        if len(_CSR_CACHE) > 8:
            _CSR_CACHE.clear()
        hit = _CSR_CACHE[key] = (CsrSupport.from_torch_sparse(G), G)
    return hit[0]
