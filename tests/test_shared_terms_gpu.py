"""RecurrentStack computes the spatial terms of each hidden state once for the two cells that read it (stack.share_plan).
The reference here is the same roll-out composed from the functional cell, which shares nothing: the stack's output
must be bitwise equal to it, and every gradient within the stack floor 1e-4 |ref| + 5e-5 mean|ref| (the shared adjoint
hop and dGs product re-associate Gs (a + b) = Gs a + Gs b)."""
import pytest
import torch

import stc_gnn_b200 as S
from stc_gnn_b200 import _lib
from stc_gnn_b200.stack import _XSideTerms, _hoistable
from stc_gnn_b200.synth import grid_csr, sf_supports

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def reference_rollout(stack, Gs, Gc, X):
    """RecurrentStack.forward with one independent cell call per step (layer 0 takes the same hoisted input terms)."""
    B, T = X.shape[0], X.shape[1]
    seq, last = [X[:, t] for t in range(T)], []
    for li, cell in enumerate(stack.encoder):
        H, outs = cell.init_hidden(B), []
        yx = _XSideTerms.apply(Gs, X) if (li == 0 and _hoistable(Gs, X, cell)) else None
        for t in range(T):
            if yx is not None:
                H = cell(Gs=Gs, Gc=Gc, Xt=seq[t], Ht_1=H, _Yx=yx[t])
            else:
                H = S.stc_cell_forward(Gs, Gc, seq[t], H, cell.gates.W, cell.gates.b, cell.candi.W, cell.candi.b,
                                       cell.Ks, cell.Kc)
            outs.append(H)
        seq = outs
        last.append(H)
    if stack.out_horizon == 0:
        return torch.stack(seq, dim=1)
    states, x, outs = last, last[-1], []
    for _ in range(stack.out_horizon):
        new, inp = [], x
        for l, cell in enumerate(stack.decoder):
            inp = S.stc_cell_forward(Gs, Gc, inp, states[l], cell.gates.W, cell.gates.b, cell.candi.W, cell.candi.b,
                                     cell.Ks, cell.Kc)
            new.append(inp)
        states, x = new, new[-1]
        outs.append(x)
    return torch.stack(outs, dim=1)


def close(got, ref, name):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    err = (got - ref).abs()
    tol = 1e-4 * ref.abs() + 5e-5 * ref.abs().mean()
    nbad = int((err > tol).sum())
    assert nbad == 0, f"{name}: {nbad}/{ref.numel()} outside the stack floor, worst {(err - tol).max().item():.3e}"


def make_case(kind, N=100, C=5, h=16, Din=1, Ks=2, layers=2, T=9, horizon=3, B=8, x_grad=False, seed=0):
    torch.manual_seed(seed)
    stack = S.RecurrentStack(N, C, Ks, 2, Din, h, layers, horizon).to(DEV)
    g = torch.Generator().manual_seed(seed + 1)
    if kind == "dense":
        if N == 100:
            Gs, Gc = sf_supports(seed=0)
        else:
            Gs, Gc = torch.rand(N, N, generator=g) / N, torch.rand(C, C, generator=g) / C
        Gs = Gs.to(DEV).requires_grad_(True)
        extra = [Gs]
    else:
        side = int(round(N ** 0.5))
        rp, ci, va = grid_csr(side, side)
        Gc = torch.rand(C, C, generator=g) / C
        vals = va.to(DEV)
        if kind == "csr_learned":
            vals = (vals * (1 + 0.2 * torch.rand(vals.shape, generator=g).to(DEV))).requires_grad_(True)
        Gs = S.CsrSupport(rp.to(DEV), ci.to(DEV), vals, side * side)
        extra = [vals] if kind == "csr_learned" else []
    Gc = Gc.to(DEV).requires_grad_(True)
    X = (torch.rand(B, T, N, C, Din, generator=g) < 0.3).float().to(DEV)
    if x_grad:
        X.requires_grad_(True)
    dOut = torch.randn(B, horizon or T, N, C, h, generator=g).to(DEV)
    leaves = list(stack.parameters()) + extra + [Gc] + ([X] if x_grad else [])
    return stack, Gs, Gc, X, dOut, leaves


def run(fn, stack, Gs, Gc, X, dOut, leaves):
    for p in leaves:
        p.grad = None
    out = fn(stack, Gs, Gc, X)
    out.backward(dOut)
    torch.cuda.synchronize()
    return out.detach().clone(), [p.grad.clone() if p.grad is not None else torch.zeros_like(p) for p in leaves]


CASES = {
    "sf": dict(kind="dense"),
    "dense_ks3": dict(kind="dense", Ks=3, T=4, horizon=2),
    "csr_const": dict(kind="csr_const", T=4, horizon=2),
    "csr_learned": dict(kind="csr_learned", T=4, horizon=2),
    "horizon0": dict(kind="dense", T=5, horizon=0),
    "layers3": dict(kind="dense", layers=3, T=3, horizon=2),
    "t1": dict(kind="dense", T=1, horizon=2),
    "x_grad": dict(kind="dense", T=4, horizon=2, x_grad=True),
    "wide": dict(kind="dense", N=64, C=8, h=64, Din=64, T=3, horizon=2, B=2),
}


@pytest.mark.parametrize("case", list(CASES))
def test_stack_equals_unshared_rollout(case):
    stack, Gs, Gc, X, dOut, leaves = make_case(**CASES[case])
    out_r, g_r = run(reference_rollout, stack, Gs, Gc, X, dOut, leaves)
    out_s, g_s = run(lambda st, a, b, c: st(a, b, c), stack, Gs, Gc, X, dOut, leaves)
    assert torch.equal(out_s, out_r), f"{case}: forward differs"
    spec = CASES[case]
    names = [n for n, _ in stack.named_parameters()] + {"dense": ["Gs"], "csr_learned": ["vals"]}.get(spec["kind"], []) \
        + ["Gc"] + (["X"] if spec.get("x_grad") else [])
    assert len(names) == len(leaves)
    for name, a, b in zip(names, g_s, g_r):
        close(a, b, f"{case} grad {name}")


def test_no_grad_forward_is_bitwise():
    stack, Gs, Gc, X, _, _ = make_case("dense", T=5, horizon=3)
    with torch.no_grad():
        a = stack(Gs, Gc, X)
        b = reference_rollout(stack, Gs, Gc, X)
    assert torch.equal(a, b)


def test_graphed_step_replays_the_shared_rollout():
    stack, Gs, Gc, X0, dOut, leaves = make_case("dense", T=4, horizon=2, seed=5)
    X1 = (torch.rand(X0.shape, generator=torch.Generator().manual_seed(9)) < 0.3).float().to(DEV)
    loss_fn = lambda X: (stack(Gs, Gc, X) * dOut).sum()
    gs = S.GraphedStep(loss_fn, [X0], leaves)
    loss_g = float(gs.replay(X1).item())
    grads_g = [p.grad.clone() for p in leaves]
    for p in leaves:
        p.grad = None
    loss_e = loss_fn(X1)
    loss_e.backward()
    assert abs(loss_g - float(loss_e.item())) <= 1e-5 * abs(float(loss_e.item()))
    for i, (a, p) in enumerate(zip(grads_g, leaves)):
        close(a, p.grad, f"graphed grad {i}")


def kinds_of_one_step(fn, stack, Gs, Gc, X, dOut, leaves):
    run(fn, stack, Gs, Gc, X, dOut, leaves)   # warm
    _lib.timing_enable(True)
    _lib.timing_collect()
    run(fn, stack, Gs, Gc, X, dOut, leaves)
    _lib.timing_enable(False)
    return {k: v[1] for k, v in _lib.timing_collect().items()}


def test_sf_launch_counts():
    """SF shape: 16 forward hops (14 shared states + 2 zero initial states), 16 adjoint hops and 16 dGs products go."""
    case = make_case("dense", B=256)
    ref = kinds_of_one_step(reference_rollout, *case)
    got = kinds_of_one_step(lambda st, a, b, c: st(a, b, c), *case)
    assert got["tc_support"] == ref["tc_support"] - 32, (got, ref)
    assert got["tc_outer"] == ref["tc_outer"] - 16, (got, ref)
    for k in set(ref) | set(got):
        if k not in ("tc_support", "tc_outer"):
            assert got.get(k) == ref.get(k), (k, got, ref)
