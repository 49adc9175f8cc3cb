"""Per-sample spatial graphs on the GPU: a CsrSupport with values [B, nnz] (one graph per input window on a shared
pattern) through the hop, the fused edge-gradient hop, the cell, the stack and the per-sample sparse graph generator.

Tolerance as everywhere: |got - ref| <= 1e-4 * |ref| + 1e-5 * mean|ref| per cell, 5e-5 * mean|ref| through a stack."""
import pytest
import torch

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from stc_gnn_b200 import _lib, cell as cell_mod
from stc_gnn_b200.synth import grid_csr
from tests import per_sample_oracle as PS
from tests import sparse_mgp_oracle as M
from tests.helpers import random_case
from tests.test_learned_csr_gpu import pattern

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
ARGS = ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")


@pytest.fixture
def deterministic():
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(was)
    _lib.sync_deterministic()


def per_sample_vals(B, vals, seed):
    """[B, nnz]: the pattern's values scaled differently in every sample (the explicit zeros stay zeros)."""
    g = torch.Generator().manual_seed(seed)
    return vals.float()[None] * (0.5 + torch.rand(B, vals.numel(), generator=g))


def kinds_of(step):
    _lib.timing_enable(True)
    _lib.timing_collect()
    step()
    torch.cuda.synchronize()
    _lib.timing_enable(False)
    return {k for k, v in _lib.timing_collect().items() if v[1]}


# ---- 1. the hop -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("width", [1, 3, 5, 64, 80, 1024, 1100])
@pytest.mark.parametrize("transpose", [True, False])
def test_hop_is_bitwise_b_single_sample_hops(width, transpose):
    B, N = 3, 300
    rowptr, col, vals = pattern(N, 8, seed=width, empty_every=7, hub=(5, 200))
    V = per_sample_vals(B, vals, width).to(DEV)
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), V, N)
    assert sup.batch == B and sup.struct().kind == _lib.SUPPORT_CSR_PER_SAMPLE
    g = torch.Generator().manual_seed(width + 1)
    X, Z = (torch.randn(B, N, width, generator=g).to(DEV) for _ in range(2))
    for kw in (dict(), dict(alpha=2.0, beta=-1.0, Z=Z)):
        Y = S.support_apply(sup, X, transpose=transpose, **kw)
        for b in range(B):
            one = sup.with_values(V[b])
            kb = {k: (v[b:b + 1] if k == "Z" else v) for k, v in kw.items()}
            assert torch.equal(Y[b:b + 1], S.support_apply(one, X[b:b + 1], transpose=transpose, **kb)), (b, kw)


# ---- 2. the edge-gradient hop ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("width", [1, 5, 64, 1100])
def test_edge_grad_hop(width):
    B, N = 3, 257
    rowptr, col, vals = pattern(N, 8, seed=width + 3, empty_every=9)
    V = per_sample_vals(B, vals, width).to(DEV)
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), V, N)
    g = torch.Generator().manual_seed(width)
    X, Z = (torch.randn(B, N, width, generator=g).to(DEV) for _ in range(2))
    A = torch.randn(B, 2, N, width, generator=g).to(DEV)[:, 1]           # batch-strided view
    buf = torch.zeros(B * sup.nnz + 64, device=DEV)
    buf[B * sup.nnz:] = 777.0
    dvals = buf[:B * sup.nnz].view(B, sup.nnz)
    Y = S.support_apply_edge_grad(sup, X, A, dvals, coef=2.0, alpha=2.0, beta=1.0, Z=Z)
    assert torch.equal(Y, S.support_apply(sup, X, transpose=False, alpha=2.0, beta=1.0, Z=Z))
    assert bool((buf[B * sup.nnz:] == 777.0).all()), "nothing past dvals[B, nnz] may be written"
    r, c = M.edge_rows(rowptr), col.long()
    ref = 2.0 * (A.double().cpu()[:, r] * X.double().cpu()[:, c]).sum(-1)
    O.assert_close(dvals.cpu(), ref, f"dvals W={width}")


def test_edge_grad_hop_deterministic_is_the_b1_call(deterministic):
    _lib.sync_deterministic()
    B, N, width = 4, 333, 48
    rowptr, col, vals = pattern(N, 8, seed=9, empty_every=5)
    V = per_sample_vals(B, vals, 9).to(DEV)
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), V, N)
    g = torch.Generator().manual_seed(1)
    X, A = (torch.randn(B, N, width, generator=g).to(DEV) for _ in range(2))
    runs = []
    for _ in range(2):
        d = torch.zeros(B, sup.nnz, device=DEV)
        S.support_apply_edge_grad(sup, X, A, d, coef=1.5)
        runs.append(d)
    assert torch.equal(runs[0], runs[1])
    for b in range(B):
        d1 = torch.zeros(sup.nnz, device=DEV)
        S.support_apply_edge_grad(sup.with_values(V[b]), X[b:b + 1], A[b:b + 1], d1, coef=1.5)
        assert torch.equal(runs[0][b], d1), b


# ---- cell helpers ----------------------------------------------------------------------------------------------------
def dev_params(t):
    return {k: t[k].float().to(DEV).requires_grad_(True) for k in ARGS}


def cell_step(sup, p, dHn, Ks, Kc, strided=False):
    """One forward + backward; returns H' and dXt.  `strided`: Xt is the encoder's [:, t] view of a [B, T, N, C, Din]
    sequence (a batch stride larger than the sample's slab)."""
    if strided:
        seq = torch.zeros((p["Xt"].shape[0], 3) + tuple(p["Xt"].shape[1:]), device=DEV)
        seq[:, 1] = p["Xt"].detach()
        seq.requires_grad_(True)
        Xt = seq[:, 1]
        assert Xt.stride(0) == 3 * Xt[0].numel()
    else:
        Xt = p["Xt"]
    Hn = S.stc_cell_forward(sup, p["Gc"], Xt, *(p[k] for k in ARGS[2:]), Ks, Kc)
    Hn.backward(dHn)
    return Hn, (seq.grad[:, 1] if strided else p["Xt"].grad)


def _cell_vs_oracle(B, N, C, Din, h, Ks, Kc, rowptr, col, vals, seed, learn=True, strided=False, w_atol=1e-5):
    V = per_sample_vals(B, vals, seed)
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=seed)
    Hn_o, g_o = PS.cell_with_grads(t, rowptr, col, V.double(), Ks, Kc)
    v = V.to(DEV).requires_grad_(learn)
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), v, N)
    dHn = t["dHn"].float().to(DEV)
    kinds = kinds_of(lambda: cell_step(sup, dev_params(t), dHn, Ks, Kc, strided))   # warm-up run, kernels recorded
    v.grad = None
    p = dev_params(t)
    Hn, dXt = cell_step(sup, p, dHn, Ks, Kc, strided)
    torch.cuda.synchronize()
    O.assert_close(Hn.detach().cpu(), Hn_o, "Hn")
    O.assert_close(dXt.cpu(), g_o["dXt"], "dXt")
    if learn:
        O.assert_close(v.grad.cpu(), g_o["dvals"], "dvals")
    for k, name in (("H", "dH"), ("bg", "dbg"), ("bc", "dbc"), ("Gc", "dGc")):
        O.assert_close(p[k].grad.cpu(), g_o[name], name)
    for k, name in (("Wg", "dWg"), ("Wc", "dWc")):
        O.assert_close(p[k].grad.cpu(), g_o[name], name, atol_scale=w_atol)
    return kinds


KERNELS_RAN = {}


# ---- 4. cell against the fp64 oracle ---------------------------------------------------------------------------------
@pytest.mark.parametrize("Ks", [1, 2, 3, 4])
@pytest.mark.parametrize("Kc", [1, 2, 3])
def test_cell_orders_match_oracle(Ks, Kc):
    B, N, C, Din, h = 3, 90, 4, 3, 8
    rowptr, col, vals = pattern(N, 6, seed=Ks * 4 + Kc, empty_every=8)
    KERNELS_RAN[f"orders Ks={Ks} Kc={Kc}"] = _cell_vs_oracle(B, N, C, Din, h, Ks, Kc, rowptr, col, vals, seed=Ks + 5 * Kc)


TIERS = {   # (B, N, C, Din, h, Ks, Kc, strided Xt): the SF tensor-core, wide-state and general FFMA convolution tiers
    "sf_tc": (4, 100, 5, 1, 16, 2, 2, True),
    "wide": (2, 64, 16, 16, 64, 2, 2, False),
    "ffma": (3, 80, 3, 2, 6, 3, 3, False),
}


@pytest.mark.parametrize("tier", list(TIERS))
@pytest.mark.parametrize("learn", [True, False])
def test_cell_tiers_match_oracle(tier, learn):
    B, N, C, Din, h, Ks, Kc, strided = TIERS[tier]
    rowptr, col, vals = pattern(N, 6, seed=len(tier), empty_every=9)
    kinds = _cell_vs_oracle(B, N, C, Din, h, Ks, Kc, rowptr, col, vals, seed=3, learn=learn, strided=strided)
    KERNELS_RAN[f"{tier} learn={learn}"] = kinds
    assert ("support_csr_grad" in kinds) == learn


def test_config3_grid4096_b4():
    rowptr, col, vals = grid_csr(64, 64)
    KERNELS_RAN["g4096"] = _cell_vs_oracle(4, 4096, 16, 1, 16, 2, 2, rowptr, col, vals, seed=11)


def test_kernels_recorded():
    """What ran in the oracle cases above, as tests/test_conv_variants_gpu.py records it."""
    for name, kinds in KERNELS_RAN.items():
        print(f"{name}: {sorted(kinds)}")
    assert all("support_csr" in k or name.startswith("orders Ks=1") for name, k in KERNELS_RAN.items())


# ---- 3. broadcast and 5. batch independence --------------------------------------------------------------------------
def _shared_vs_per_sample(t, rowptr, col, vals, B, N):
    shared_v = vals.float().to(DEV).requires_grad_(True)
    ps_v = shared_v.detach()[None].repeat(B, 1).requires_grad_(True)
    out = []
    for v in (shared_v, ps_v):
        sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), v, N)
        p = dev_params(t)
        Hn = S.stc_cell_forward(sup, *(p[k] for k in ARGS), 3, 2)
        Hn.backward(t["dHn"].float().to(DEV))
        torch.cuda.synchronize()
        out.append((Hn.detach(), {k: x.grad for k, x in p.items()}, v.grad))
    return out


def test_broadcast_equals_shared_support():
    B, N, C, Din, h = 4, 120, 5, 2, 16
    rowptr, col, vals = pattern(N, 6, seed=21, empty_every=7)
    t = random_case(B, N, C, Din, h, 3, 2, seed=21)
    (H1, g1, dv1), (H2, g2, dv2) = _shared_vs_per_sample(t, rowptr, col, vals, B, N)
    assert torch.equal(H1, H2)
    ref = dv1.double().cpu()
    err, tol = (dv2.sum(0).double().cpu() - ref).abs(), 1e-4 * ref.abs() + 5e-5 * ref.abs().mean()
    assert bool((err <= tol).all())


def test_broadcast_deterministic_bitwise(deterministic):
    B, N, C, Din, h = 4, 120, 5, 2, 16
    rowptr, col, vals = pattern(N, 6, seed=22, empty_every=7)
    t = random_case(B, N, C, Din, h, 3, 2, seed=22)
    (H1, g1, dv1), (H2, g2, dv2) = _shared_vs_per_sample(t, rowptr, col, vals, B, N)
    assert torch.equal(H1, H2)
    for k in ("Xt", "H", "Wg", "Wc", "Gc"):
        assert torch.equal(g1[k], g2[k]), k


def test_batch_independence():
    B, N, C, Din, h = 8, 150, 5, 1, 16
    rowptr, col, vals = pattern(N, 6, seed=23)
    t = random_case(B, N, C, Din, h, 2, 2, seed=23)
    V = per_sample_vals(B, vals, 23).to(DEV)
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), V, N)
    p = {k: t[k].float().to(DEV) for k in ARGS}
    Hn = S.stc_cell_forward(sup, *(p[k] for k in ARGS), 2, 2)
    for b in (0, B // 2, B - 1):
        one = {k: (x[b:b + 1] if k in ("Xt", "H") else x) for k, x in p.items()}
        Hb = S.stc_cell_forward(sup.with_values(V[b]), *(one[k] for k in ARGS), 2, 2)
        assert float((Hn[b:b + 1] - Hb).abs().max()) <= 1e-6, b


# ---- 6. value handling and 7. forward-only -----------------------------------------------------------------------------
@pytest.mark.parametrize("inplace", [True, False])
def test_value_handling(monkeypatch, inplace):
    monkeypatch.setattr(cell_mod, "INPLACE_LEAF_GRADS", inplace)
    B, N, C, Din, h = 3, 70, 4, 2, 8
    rowptr, col, vals = pattern(N, 5, seed=31)
    t = random_case(B, N, C, Din, h, 2, 2, seed=31)
    leaf = torch.nn.Parameter(per_sample_vals(B, vals, 31).to(DEV))
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), leaf, N)
    p = {k: t[k].float().to(DEV) for k in ARGS}
    run = lambda s: S.stc_cell_forward(s, *(p[k] for k in ARGS), 2, 2)
    dHn = t["dHn"].float().to(DEV)
    run(sup).backward(dHn)
    g_leaf = leaf.grad.clone()
    assert g_leaf.shape == (B, sup.nnz)
    with torch.no_grad():
        leaf.mul_(1.5)               # an in-place update is seen by the next forward
    fresh = S.CsrSupport(rowptr.to(DEV), col.to(DEV), leaf.detach().clone(), N)
    assert torch.equal(run(sup).detach(), run(fresh))
    raw = torch.nn.Parameter(torch.randn(B, sup.nnz, device=DEV) * 0.1)   # non-leaf values
    nl = sup.with_values(torch.nn.functional.softplus(raw))
    run(nl).backward(dHn)
    assert raw.grad is not None and raw.grad.shape == (B, sup.nnz) and bool(raw.grad.abs().sum() > 0)


def test_forward_only_is_bitwise_the_training_forward():
    B, N, C, Din, h = 3, 90, 5, 1, 16
    rowptr, col, vals = pattern(N, 6, seed=41)
    t = random_case(B, N, C, Din, h, 3, 2, seed=41)
    leaf = per_sample_vals(B, vals, 41).to(DEV).requires_grad_(True)
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), leaf, N)
    p = dev_params(t)
    H_train = S.stc_cell_forward(sup, *(p[k] for k in ARGS), 3, 2).detach()
    cell_mod._SIZES.clear()
    with torch.no_grad():
        H_fo = S.stc_cell_forward(sup, *(p[k] for k in ARGS), 3, 2)
    assert any(k[0] == "fwd_only" for k in cell_mod._SIZES), "no_grad must take stc_cell_fwd_only"
    assert torch.equal(H_train, H_fo)


# ---- 8. stack, 9. graph replay, 10. deterministic training steps -------------------------------------------------------
def _stack_case(seed=0, B=3, N=49, C=4, h=8, T=4, horizon=2):
    torch.manual_seed(seed)
    stack = S.RecurrentStack(N, C, 2, 2, 1, h, 2, horizon).to(DEV)
    gen = S.SparseGraphGenerator(C, 6).to(DEV)
    side = int(round(N ** 0.5))
    rowptr, col, _ = grid_csr(side, side)
    pat = S.CsrSupport(rowptr.to(DEV), col.to(DEV), torch.zeros(col.numel(), device=DEV), N)
    g = torch.Generator().manual_seed(seed + 1)
    Gc = (torch.rand(C, C, generator=g) / C).to(DEV).requires_grad_(True)
    X = torch.randn(B, T, N, C, 1, generator=g).to(DEV)
    dOut = torch.randn(B, horizon, N, C, h, generator=g).to(DEV)
    return stack, gen, pat, Gc, X, dOut, (rowptr, col)


def test_stack_on_generated_per_sample_support_matches_oracle():
    stack, gen, pat, Gc, X, dOut, (rowptr, col) = _stack_case()
    Gs = gen(X[..., 0], pat, per_sample=True)
    assert Gs.batch == X.shape[0]
    out = stack(Gs, Gc, X)
    # the fp64 oracle stack on the same generated values
    P = Gs.vals.detach().double().cpu()
    Gd = PS.dense_batch(rowptr, col, P, pat.N)
    cell_fn = lambda G, *a: O.stc_cell(None, *a, spatial_terms_fn=PS.per_sample_terms(G, a[7]))
    enc = [O.CellParams(*(x.detach().double().cpu() for x in (c.gates.W, c.gates.b, c.candi.W, c.candi.b)))
           for c in stack.encoder]
    dec = [O.CellParams(*(x.detach().double().cpu() for x in (c.gates.W, c.gates.b, c.candi.W, c.candi.b)))
           for c in stack.decoder]
    ref = O.stack_forward(Gd, Gc.detach().double().cpu(), X.double().cpu(), enc, dec, 2, 2, 2, cell_fn=cell_fn)
    err = (out.detach().double().cpu() - ref).abs()
    assert bool((err <= 1e-4 * ref.abs() + 5e-5 * ref.abs().mean()).all())
    out.backward(dOut)
    assert gen.params_S["Wu"].grad is not None and bool(gen.params_S["Wu"].grad.abs().sum() > 0)


def test_stack_shares_terms_with_a_per_sample_support():
    from tests.test_shared_terms_gpu import reference_rollout
    stack, gen, pat, Gc, X, dOut, _ = _stack_case(seed=2)
    with torch.no_grad():
        Gs = gen(X[..., 0], pat, per_sample=True)
    Gs = Gs.with_values(Gs.vals.clone().requires_grad_(True))
    leaves = list(stack.parameters()) + [Gs.vals, Gc]

    def run(fn):
        for q in leaves:
            q.grad = None
        out = fn()
        out.backward(dOut)
        torch.cuda.synchronize()
        return out.detach(), [q.grad.clone() for q in leaves]

    def count(fn):
        run(fn)
        _lib.timing_enable(True)
        _lib.timing_collect()
        res = run(fn)
        _lib.timing_enable(False)
        return res, {k: v[1] for k, v in _lib.timing_collect().items()}

    (o_r, g_r), k_r = count(lambda: reference_rollout(stack, Gs, Gc, X))
    (o_s, g_s), k_s = count(lambda: stack(Gs, Gc, X))
    assert torch.equal(o_s, o_r)
    for a, b in zip(g_s, g_r):
        err = (a.double() - b.double()).abs()
        assert bool((err <= 1e-4 * b.double().abs() + 5e-5 * b.double().abs().mean()).all())
    assert k_s["support_csr"] < k_r["support_csr"], (k_s, k_r)
    assert k_s["support_csr_grad"] < k_r["support_csr_grad"], (k_s, k_r)


def test_graphed_step_with_the_per_sample_generator():
    stack, gen, pat, Gc, X0, dOut, _ = _stack_case(seed=3)
    X1 = torch.randn(X0.shape, generator=torch.Generator().manual_seed(8)).to(DEV)
    leaves = list(stack.parameters()) + list(gen.parameters()) + [Gc]
    loss_fn = lambda X: (stack(gen(X[..., 0], pat, per_sample=True), Gc, X) * dOut).sum()
    gs = S.GraphedStep(loss_fn, [X0], leaves)
    loss_g = float(gs.replay(X1).item())
    grads_g = [q.grad.clone() for q in leaves]
    for q in leaves:
        q.grad = None
    loss_e = loss_fn(X1)
    loss_e.backward()
    assert abs(loss_g - float(loss_e.item())) <= 1e-5 * abs(float(loss_e.item()))
    for a, q in zip(grads_g, leaves):
        err = (a.double() - q.grad.double()).abs()
        assert bool((err <= 1e-4 * q.grad.double().abs() + 5e-5 * q.grad.double().abs().mean()).all())


def test_deterministic_training_steps_are_bitwise(deterministic):
    """(cuBLAS inside the generator needs CUBLAS_WORKSPACE_CONFIG in this mode, so the per-sample values are a leaf.)"""
    stack, gen, pat, Gc, X, dOut, _ = _stack_case(seed=4)
    with torch.no_grad():
        P = gen(X[..., 0], pat, per_sample=True).vals
    Gs = pat.with_values(P.clone().requires_grad_(True))
    leaves = list(stack.parameters()) + [Gs.vals, Gc]
    runs = []
    for _ in range(2):
        for q in leaves:
            q.grad = None
        out = stack(Gs, Gc, X)
        out.backward(dOut)
        torch.cuda.synchronize()
        runs.append([out.detach().clone()] + [q.grad.clone() for q in leaves])
    for a, b in zip(*runs):
        assert torch.equal(a, b)


# ---- 11. the generator -----------------------------------------------------------------------------------------------
def _knn_pattern_with_empty_rows_and_self_loops(N):
    rowptr, col = M.random_pattern(N, 8, seed=5, empty_every=7, self_loop_every=3)
    return rowptr, col


@pytest.mark.parametrize("pat", ["grid64", "random"])
def test_generator_is_bitwise_each_window_alone(pat):
    if pat == "grid64":
        rowptr, col, _ = grid_csr(64, 64)
    else:
        rowptr, col = _knn_pattern_with_empty_rows_and_self_loops(500)
    N = rowptr.numel() - 1
    B, T, C, hg = 4, 6, 5, 16
    torch.manual_seed(0)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    patt = S.CsrSupport(rowptr.to(DEV), col.to(DEV), torch.zeros(col.numel(), device=DEV), N)
    X = torch.randn(B, T, N, C, generator=torch.Generator().manual_seed(1)).to(DEV).requires_grad_(True)
    Gs = gen(X, patt, per_sample=True)
    assert Gs.batch == B and Gs.vals.shape == (B, patt.nnz) and Gs.vals.requires_grad
    for b in range(B):
        assert torch.equal(Gs.vals[b].detach(), gen(X[b:b + 1].detach(), patt).vals.detach()), b
    if pat == "grid64":
        return
    # gradients (on the smaller pattern: few scores lie close enough to 0 for fp32 and fp64 to disagree on the relu) into Wu, Wv and X_seq against fp64 autograd of the restatement
    dP = torch.randn(B, patt.nnz, generator=torch.Generator().manual_seed(2)).to(DEV)
    (Gs.vals * dP).sum().backward()
    Xd = X.detach().double().cpu().requires_grad_(True)
    Wu = gen.params_S["Wu"].detach().double().cpu().requires_grad_(True)
    Wv = gen.params_S["Wv"].detach().double().cpu().requires_grad_(True)
    P = PS.generator(Xd, Wu, Wv, gen.alpha, rowptr, col)
    O.assert_close(Gs.vals.detach().cpu(), P.detach(), "P")
    (P * dP.double().cpu()).sum().backward()
    O.assert_close(gen.params_S["Wu"].grad.cpu(), Wu.grad, "dWu")
    O.assert_close(gen.params_S["Wv"].grad.cpu(), Wv.grad, "dWv")
    O.assert_close(X.grad.cpu(), Xd.grad, "dX_seq")
    with torch.no_grad():
        c = gen(X, patt, per_sample=True)
    assert not c.vals.requires_grad and not c.learnable and c.batch == B
    assert torch.equal(c.vals, Gs.vals.detach())


# ---- 12. two ranks over gloo on one GPU ---------------------------------------------------------------------------------
def _dp_worker(rank, world, port, q):
    import os
    import traceback
    import torch.distributed as dist
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        stack, gen, pat, Gc, X, dOut, _ = _stack_case(seed=6, B=4)
        leaves = list(stack.parameters()) + list(gen.parameters()) + [Gc]

        def step(Xs, dO):
            for p_ in leaves:
                p_.grad = None
            Gs = gen(Xs[..., 0], pat, per_sample=True)
            out = stack(Gs, Gc, Xs)
            out.backward(dO)
            return out.detach()

        out_g = step(X, dOut)                 # the single-process global batch, on every rank
        grads_g = [p_.grad.clone() for p_ in leaves]
        calls = []
        real = {n: getattr(dist, n) for n in ("all_reduce", "all_gather", "all_gather_into_tensor", "all_to_all",
                                              "all_to_all_single", "broadcast", "reduce_scatter")}
        for n, f in real.items():
            setattr(dist, n, (lambda n_, f_: (lambda *a, **k: (calls.append(n_), f_(*a, **k))[1]))(n, f))
        out_s = step(S.dp.shard_batch(X, rank, world), S.dp.shard_batch(dOut, rank, world))
        torch.cuda.synchronize()
        assert calls == [], f"the generator and the stack made collective calls: {calls}"
        for n, f in real.items():
            setattr(dist, n, f)
        lo, hi = S.dp.shard_bounds(X.shape[0], rank, world)
        assert float((out_s - out_g[lo:hi]).abs().max()) <= 1e-6
        S.dp.GradBucket([p_ for p_ in leaves]).allreduce()
        for a, p_ in zip(grads_g, leaves):
            err = (p_.grad.double() - a.double()).abs()
            assert bool((err <= 1e-4 * a.double().abs() + 5e-5 * a.double().abs().mean()).all())
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, None))
    except Exception:  # pragma: no cover - reported by the parent
        q.put((rank, traceback.format_exc()))


def test_two_ranks_gloo_batch_shards():
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    try:
        results = [q.get(timeout=600) for _ in procs]
    finally:
        for pr in procs:
            pr.join(timeout=60)
            if pr.is_alive():
                pr.terminate()
                pr.join()
    for rank, err in results:
        assert err is None, f"rank {rank}:\n{err}"


# ---- 13. errors ----------------------------------------------------------------------------------------------------------
def test_errors():
    B, N, C = 3, 40, 4
    rowptr, col, vals = pattern(N, 4, seed=51)
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), per_sample_vals(B, vals, 51).to(DEV), N)
    t = random_case(B + 1, N, C, 1, 8, 2, 2, seed=51)
    p = {k: t[k].float().to(DEV) for k in ARGS}
    with pytest.raises(RuntimeError, match=r"B = 3.*B = 4"):
        S.stc_cell_forward(sup, *(p[k] for k in ARGS), 2, 2)
    X = torch.randn(B, N, 8, device=DEV)
    rows = torch.arange(5, dtype=torch.int32, device=DEV)
    with pytest.raises(RuntimeError, match="per-sample"):
        S.support_apply(sup, X, out=torch.empty_like(X), rows=rows)
    with pytest.raises(RuntimeError, match="per-sample"):
        S.support_apply_edge_grad(sup, X, X, torch.zeros(B, sup.nnz, device=DEV), out=torch.empty_like(X), rows=rows)
    gen = S.SparseGraphGenerator(C, 4).to(DEV)
    Xs = torch.randn(B, 3, N, C, device=DEV)
    with pytest.raises(RuntimeError, match="per-sample top-k"):
        gen(Xs, k=4, per_sample=True)
    with pytest.raises(RuntimeError, match="per-sample top-k"):
        gen(Xs, k=4, partition=S.halo.RowPartition(N, 0, 1), per_sample=True)
    with pytest.raises(RuntimeError, match="needs no communication"):
        gen(Xs, sup, group=object(), per_sample=True)
    with pytest.raises(RuntimeError, match="needs no communication"):
        gen(Xs, sup, average=True, per_sample=True)
    with pytest.raises(RuntimeError, match="per-sample"):
        S.halo.PartitionedSupport.from_csr_support(sup, 0, 1)
    ps = S.halo.PartitionedSupport.__new__(S.halo.PartitionedSupport)   # (the checks run before any of its state)
    ps.nnz = sup.nnz
    with pytest.raises(RuntimeError, match="row-partitioned"):
        gen(Xs, ps, per_sample=True)
    with pytest.raises(RuntimeError, match="per-sample"):
        ps.with_values(torch.zeros(B, ps.nnz, device=DEV))
    lib = _lib.load()
    st = sup.struct()
    Y = torch.empty_like(X)
    status = lib.stc_support_apply_rows(st, N, B, 8, 1, X.data_ptr(), N * 8, None, N * 8, Y.data_ptr(), 1.0, 0.0,
                                        rows.data_ptr(), 5, torch.cuda.current_stream().cuda_stream)
    assert status == -2 and b"STC_SUPPORT_CSR_PER_SAMPLE" in lib.stc_last_error()
