"""Learnable edge values of a CSR spatial support on the GPU: the fused adjoint hop (stc_support_apply_edge_grad), the
cell and the stack against the fp64 oracle, the ABI's clearing of the [nnz] gradient, non-leaf values, in-place
updates and CUDA-graph replay.

Tolerance as everywhere: |got - ref| <= 1e-4 * |ref| + 1e-5 * mean|ref| per cell, 5e-5 * mean|ref| through a stack."""
import pytest
import torch

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from tests.helpers import oracle_cell_with_grads, random_case
from tests.learned_csr_oracle import stc_cell_edge_grad

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def pattern(N, deg, seed, empty_every=0, hub=None, zero_frac=0.15):
    """CSR (rowptr, col, vals) host tensors: distinct sorted neighbours per row, rows with no edge (every
    `empty_every`-th), optionally one row `hub` linked to `hub[1]` nodes, and a fraction of edges stored as 0."""
    g = torch.Generator().manual_seed(seed)
    rows = []
    for n in range(N):
        d = int(torch.randint(1, deg + 1, (1,), generator=g))
        if empty_every and n % empty_every == 1:
            d = 0
        if hub is not None and n == hub[0]:
            d = hub[1]
        rows.append(torch.sort(torch.randperm(N, generator=g)[:d]).values)
    col = torch.cat(rows).to(torch.int32)
    rowptr = torch.zeros(N + 1, dtype=torch.int32)
    rowptr[1:] = torch.cumsum(torch.tensor([r.numel() for r in rows]), 0)
    vals = (torch.rand(col.numel(), generator=g) + 0.5) / deg
    vals[torch.rand(col.numel(), generator=g) < zero_frac] = 0.0
    return rowptr, col, vals


def edge_rows(rowptr):
    return torch.repeat_interleave(torch.arange(rowptr.numel() - 1), (rowptr[1:] - rowptr[:-1]).long())


def dense_of(rowptr, col, vals, N):
    G = torch.zeros(N, N, dtype=torch.float64)
    G.index_put_((edge_rows(rowptr), col.long()), vals.double(), accumulate=True)
    return G


def learnable(rowptr, col, vals, N):
    v = torch.nn.Parameter(vals.float().to(DEV))
    return S.CsrSupport(rowptr.to(DEV), col.to(DEV), v, N), v


# ---- 1. the fused hop on its own --------------------------------------------------------------------------------
@pytest.mark.parametrize("width", [1, 3, 5, 64, 512, 1024])
@pytest.mark.parametrize("B", [1, 3])
def test_fused_hop_matches_torch_and_the_plain_hop(width, B):
    N = 400
    rowptr, col, vals = pattern(N, 9, seed=width + B, empty_every=11, hub=(17, 320))
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), vals.to(DEV), N)
    g = torch.Generator().manual_seed(width * 7 + B)
    X = torch.randn(B, N, width, generator=g).to(DEV)
    Z = torch.randn(B, N, width, generator=g).to(DEV)
    A_big = torch.randn(B, 2, N, width, generator=g).to(DEV)
    A = A_big[:, 1]                                      # per-sample slab contiguous, batch stride 2 * N * width
    assert B == 1 or A.stride(0) == 2 * N * width
    coef = 2.0
    buf = torch.full((sup.nnz + 64,), 0.0, device=DEV)
    buf[sup.nnz:] = 12345.0                              # canary after dvals[nnz]
    dvals = buf[:sup.nnz]
    Y = S.support_apply_edge_grad(sup, X, A, dvals, coef=coef, alpha=coef, beta=1.0, Z=Z)
    Y_plain = S.support_apply(sup, X, transpose=False, alpha=coef, beta=1.0, Z=Z)
    torch.cuda.synchronize()
    assert torch.equal(Y, Y_plain), "the fused hop must write exactly what the plain adjoint hop writes"
    assert bool((buf[sup.nnz:] == 12345.0).all()), "nothing past dvals[nnz] may be written"
    r, c = edge_rows(rowptr), col.long()
    Ad, Xd = A.double().cpu(), X.double().cpu()
    ref = coef * (Ad[:, r] * Xd[:, c]).sum(dim=(0, 2))
    O.assert_close(dvals.cpu(), ref, f"dvals W={width} B={B}")
    # a second call adds to dvals
    S.support_apply_edge_grad(sup, X, A, dvals, coef=coef, alpha=coef, beta=1.0, Z=Z)
    O.assert_close(dvals.cpu(), 2 * ref, "dvals after a second call")


# ---- 2. cell forward + every gradient against the fp64 oracle ----------------------------------------------------
def _cell_vs_oracle(B, N, C, Din, h, Ks, Kc, rowptr, col, vals, seed, w_atol=1e-5):
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, activation=None)
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=seed)
    t["Gs"] = dense_of(rowptr, col, vals, N)
    Hn_o, g_o = oracle_cell_with_grads(t, cfg)
    sup, v = learnable(rowptr, col, vals, N)
    dev = lambda k: t[k].float().to(DEV).requires_grad_(True)
    p = {k: dev(k) for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")}
    Hn = S.stc_cell_forward(sup, p["Gc"], p["Xt"], p["H"], p["Wg"], p["bg"], p["Wc"], p["bc"], Ks, Kc)
    Hn.backward(t["dHn"].float().to(DEV))
    with torch.no_grad():   # the same cell on the detached (constant) values: the forward must be bit-identical
        const = S.CsrSupport(rowptr.to(DEV), col.to(DEV), vals.float().to(DEV), N)
        Hc = S.stc_cell_forward(const, *(p[k].detach() for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")), Ks, Kc)
    torch.cuda.synchronize()
    assert torch.equal(Hn.detach(), Hc), "H' must not depend on whether the values are learnable"
    O.assert_close(Hn.detach().cpu(), Hn_o, "Hn")
    O.assert_close(v.grad.cpu(), g_o["dGs"][edge_rows(rowptr), col.long()], "dvals")
    for k, name in (("Xt", "dXt"), ("H", "dH"), ("bg", "dbg"), ("bc", "dbc"), ("Gc", "dGc")):
        O.assert_close(p[k].grad.cpu(), g_o[name], name)
    for k, name in (("Wg", "dWg"), ("Wc", "dWc")):
        O.assert_close(p[k].grad.cpu(), g_o[name], name, atol_scale=w_atol)


@pytest.mark.parametrize("shape", [(2, 64, 4, 3, 8, 2, 2), (3, 200, 8, 16, 16, 4, 2), (1, 50, 5, 1, 16, 3, 3),
                                   (2, 64, 4, 3, 8, 1, 2)])
def test_cell_with_learnable_csr_matches_oracle(shape):
    B, N, C, Din, h, Ks, Kc = shape
    rowptr, col, vals = pattern(N, 6, seed=sum(shape), empty_every=9)
    _cell_vs_oracle(B, N, C, Din, h, Ks, Kc, rowptr, col, vals, seed=sum(shape))


def test_config3_grid4096_learnable_csr_cell():
    """N = 4096 grid (8-neighbour), C = 16, F = 64: the config 3 case with learnable, non-uniform edge values."""
    from stc_gnn_b200.synth import grid_csr
    rowptr, col, vals = grid_csr(64, 64)
    vals = vals * (0.5 + torch.rand(vals.numel(), generator=torch.Generator().manual_seed(7)))
    # dW sums 65,536 rows: the floor test_config3_grid4096_f64_csr_cell states for it (3e-5 x mean|ref|)
    _cell_vs_oracle(1, 4096, 16, 64, 64, 2, 2, rowptr, col, vals, seed=7, w_atol=3e-5)


# ---- 3. the ABI clears nnz floats, not N*N ------------------------------------------------------------------------
def test_abi_cell_bwd_clears_the_edge_gradient():
    from stc_gnn_b200 import _lib
    lib = _lib.load()
    B, N, C, Din, h, Ks, Kc = 2, 40, 3, 4, 8, 3, 2
    rowptr, col, vals = pattern(N, 5, seed=3)
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), vals.to(DEV), N)
    t = {k: (v.float().to(DEV) if v is not None else None) for k, v in random_case(B, N, C, Din, h, Ks, Kc, seed=3).items()}
    dims = _lib.StcDims(B, N, C, Din, h, Ks, Kc, 0, 1)
    saved = torch.empty(lib.stc_cell_saved_bytes(dims) // 4, device=DEV)
    scratch = torch.empty(lib.stc_cell_bwd_scratch_bytes(dims) // 4, device=DEV)
    Hn = torch.empty(B, N, C, h, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    gs = sup.struct()
    _lib.check(lib.stc_cell_fwd(dims, gs, t["Gc"].data_ptr(), t["Xt"].data_ptr(), N * C * Din, t["H"].data_ptr(),
                                t["Wg"].data_ptr(), t["bg"].data_ptr(), t["Wc"].data_ptr(), t["bc"].data_ptr(),
                                Hn.data_ptr(), saved.data_ptr(), saved.numel() * 4, st), "fwd")
    P = (Din + h) * Ks * Kc
    g = {k: torch.empty(*s, device=DEV) for k, s in (("dX", (B, N, C, Din)), ("dH", (B, N, C, h)), ("dWg", (P, 2 * h)),
                                                      ("dbg", (2 * h,)), ("dWc", (P, h)), ("dbc", (h,)), ("dGc", (C, C)))}
    buf = torch.full((sup.nnz + 256,), 7.0, device=DEV)   # garbage in dvals, a canary behind it

    def bwd(accumulate):
        _lib.check(lib.stc_cell_bwd(dims, gs, t["Gc"].data_ptr(), t["Xt"].data_ptr(), N * C * Din, t["H"].data_ptr(),
                                    t["Wg"].data_ptr(), t["Wc"].data_ptr(), t["dHn"].data_ptr(), g["dX"].data_ptr(),
                                    g["dH"].data_ptr(), g["dWg"].data_ptr(), g["dbg"].data_ptr(), g["dWc"].data_ptr(),
                                    g["dbc"].data_ptr(), buf.data_ptr(), g["dGc"].data_ptr(), accumulate,
                                    saved.data_ptr(), saved.numel() * 4, scratch.data_ptr(), scratch.numel() * 4, st), "bwd")

    bwd(0)
    once = buf[:sup.nnz].clone()
    bwd(0)
    torch.cuda.synchronize()
    O.assert_close(buf[:sup.nnz].cpu(), once.cpu(), "dvals after two overwriting calls")
    assert bool((buf[sup.nnz:] == 7.0).all()), "only nnz floats are cleared"
    bwd(1)
    O.assert_close(buf[:sup.nnz].cpu(), 2 * once.cpu(), "accumulating call adds")
    ref = stc_cell_edge_grad(torch.sparse_csr_tensor(rowptr.long(), col.long(), vals.double(), size=(N, N)),
                             *(t[k].double().cpu() for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")), Ks, Kc,
                             t["dHn"].double().cpu())
    O.assert_close(once.cpu(), ref, "dvals vs oracle")


# ---- 4. a leaf parameter through a RecurrentStack roll-out ---------------------------------------------------------
def _stack_case(seed):
    N, C, Ks, Kc, Din, h, layers, horizon, B, T = 30, 3, 3, 2, 1, 8, 2, 2, 2, 3
    torch.manual_seed(seed)
    stack = S.RecurrentStack(N, C, Ks, Kc, Din, h, layers, horizon).to(DEV)
    g = torch.Generator().manual_seed(seed)
    rowptr, col, vals = pattern(N, 5, seed=seed, empty_every=8)
    Gc = (torch.rand(C, C, generator=g) / C).to(DEV)
    X = torch.randn(B, T, N, C, Din, generator=g).to(DEV)
    dOut = torch.randn(B, horizon, N, C, h, generator=g).to(DEV)
    return stack, rowptr, col, vals, Gc, X, dOut


def _oracle_stack_dvals(stack, rowptr, col, vals, Gc, X, dOut, N):
    Gs = dense_of(rowptr, col, vals, N).requires_grad_(True)
    cp = lambda c: O.CellParams(c.gates.W.detach().double().cpu(), c.gates.b.detach().double().cpu(),
                                c.candi.W.detach().double().cpu(), c.candi.b.detach().double().cpu())
    enc, dec = [cp(c) for c in stack.encoder], [cp(c) for c in stack.decoder]
    cell0 = stack.encoder[0]
    out = O.stack_forward(Gs, Gc.double().cpu(), X.double().cpu(), enc, dec, stack.out_horizon, cell0.Ks, cell0.Kc)
    out.backward(dOut.double().cpu())
    return out.detach(), Gs.grad[edge_rows(rowptr), col.long()]


def stack_chk(got, ref, name):
    O.assert_close(got.detach().cpu(), ref, name, atol_scale=5e-5)   # the stack-level floor


def test_leaf_values_through_a_stack_rollout():
    stack, rowptr, col, vals, Gc, X, dOut = _stack_case(21)
    N = 30
    sup, v = learnable(rowptr, col, vals, N)
    out = stack(sup, Gc, X)
    out.backward(dOut)
    torch.cuda.synchronize()
    out_o, dv_o = _oracle_stack_dvals(stack, rowptr, col, vals, Gc, X, dOut, N)
    O.assert_close(out.detach().cpu(), out_o, "stack out")
    stack_chk(v.grad, dv_o, "stack dvals")
    first = v.grad.clone()
    stack(sup, Gc, X).backward(dOut)                 # a second backward adds into .grad
    torch.cuda.synchronize()
    stack_chk(v.grad, 2 * first.double(), "stack dvals after a second backward")


# ---- 5. non-leaf values ------------------------------------------------------------------------------------------
def test_non_leaf_values_and_autograd_grad(monkeypatch):
    from stc_gnn_b200 import cell as cellmod
    B, N, C, Din, h, Ks, Kc = 2, 48, 4, 3, 8, 3, 2
    rowptr, col, vals = pattern(N, 6, seed=5, zero_frac=0.0)
    raw0 = torch.log(torch.expm1(vals.double())).float()          # softplus(raw0) == vals
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=5)
    f = lambda k: t[k].float().to(DEV)
    args = [f(k) for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")]
    base = S.CsrSupport(rowptr.to(DEV), col.to(DEV), vals.to(DEV), N)
    raw = torch.nn.Parameter(raw0.to(DEV))
    vv = torch.nn.functional.softplus(raw)
    sup = base.with_values(vv)
    Hn = S.stc_cell_forward(sup, *args, Ks, Kc)
    Hn.backward(f("dHn"))
    torch.cuda.synchronize()
    Gs_ref = dense_of(rowptr, col, torch.nn.functional.softplus(raw0.double()), N)
    t["Gs"] = Gs_ref
    Hn_o, g_o = oracle_cell_with_grads(t, dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc))
    r, c = edge_rows(rowptr), col.long()
    dv_o = g_o["dGs"][r, c]
    O.assert_close(Hn.detach().cpu(), Hn_o, "Hn with_values")
    O.assert_close(raw.grad.cpu(), dv_o * torch.sigmoid(raw0.double()), "d raw")
    # torch.autograd.grad w.r.t. a leaf needs the returned form of the gradient
    monkeypatch.setattr(cellmod, "INPLACE_LEAF_GRADS", False)
    leaf_sup, leaf = learnable(rowptr, col, vv.detach().cpu(), N)
    loss = (S.stc_cell_forward(leaf_sup, *args, Ks, Kc) * f("dHn")).sum()
    (gv,) = torch.autograd.grad(loss, leaf)
    assert leaf.grad is None
    O.assert_close(gv.cpu(), dv_o, "autograd.grad dvals")


# ---- 6. an in-place update is seen by the next forward ------------------------------------------------------------
def test_inplace_update_then_second_forward():
    B, N, C, Din, h, Ks, Kc = 2, 56, 4, 2, 8, 3, 2
    rowptr, col, vals = pattern(N, 6, seed=6)
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=6)
    f = lambda k: t[k].float().to(DEV)
    args = [f(k) for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")]
    sup, v = learnable(rowptr, col, vals, N)
    S.stc_cell_forward(sup, *args, Ks, Kc).backward(f("dHn"))
    with torch.no_grad():                                        # one SGD step, in place
        v.sub_(0.5 * v.grad / v.grad.abs().max() * v.abs().max())
    v.grad = None
    Hn = S.stc_cell_forward(sup, *args, Ks, Kc)
    Hn.backward(f("dHn"))
    torch.cuda.synchronize()
    t["Gs"] = dense_of(rowptr, col, v.detach().cpu(), N)
    Hn_o, g_o = oracle_cell_with_grads(t, dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc))
    O.assert_close(Hn.detach().cpu(), Hn_o, "Hn after the update")
    O.assert_close(v.grad.cpu(), g_o["dGs"][edge_rows(rowptr), col.long()], "dvals after the update")


# ---- 7. CUDA-graph replay ------------------------------------------------------------------------------------------
def test_graphed_step_with_learnable_csr_support():
    stack, rowptr, col, vals, Gc, X0, _ = _stack_case(31)
    sup, v = learnable(rowptr, col, vals, 30)
    params = list(stack.parameters()) + [v]
    X1 = torch.randn(X0.shape, generator=torch.Generator().manual_seed(32)).to(DEV)
    loss_fn = lambda X: stack(sup, Gc, X).square().mean()
    gs = S.GraphedStep(loss_fn, [X0], params)
    with torch.no_grad():
        v.mul_(1.25)                         # an in-place update after capture: the replay must re-gather t_vals
    loss_g = float(gs.replay(X1).item())
    grads_g = [p.grad.clone() for p in params]
    for p in params:
        p.grad = None
    loss_e = loss_fn(X1)
    loss_e.backward()
    assert abs(loss_g - float(loss_e.item())) <= 1e-5 * abs(float(loss_e.item()))
    for i, (a, b) in enumerate(zip(grads_g, [p.grad for p in params])):
        O.assert_close(a.cpu(), b.double().cpu(), f"graphed grad {i}")


# ---- 8. a constant support never launches the gradient variant -----------------------------------------------------
def test_constant_support_launches_no_gradient_hop():
    from stc_gnn_b200 import _lib
    B, N, C, Din, h, Ks, Kc = 2, 64, 4, 3, 8, 3, 2
    rowptr, col, vals = pattern(N, 6, seed=8)
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=8)
    f = lambda k: t[k].float().to(DEV).requires_grad_(True)

    def kinds_of(sup):
        args = [f(k) for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")]
        _lib.timing_enable(True)
        _lib.timing_collect()
        S.stc_cell_forward(sup, *args, Ks, Kc).backward(f("dHn").detach())
        torch.cuda.synchronize()
        _lib.timing_enable(False)
        return _lib.timing_collect()

    const = kinds_of(S.CsrSupport(rowptr.to(DEV), col.to(DEV), vals.to(DEV), N))
    assert "support_csr_grad" not in const and const["support_csr"][1] > 0, const
    learned = kinds_of(learnable(rowptr, col, vals, N)[0])
    assert learned["support_csr_grad"][1] == 3 * (Ks - 1), learned   # every adjoint hop of the three chains
