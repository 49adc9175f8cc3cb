"""The adjoint hop and the dGs product of a dense support with N <= 112 run as one kernel (tc_support_adj) when a cell
call's side lanes are inactive, and as the pair tc_support + tc_outer when they are active.  `set_concurrency(0)` and
`(1)` select the two on the same inputs: the hop half is bitwise the pair's, so d_h_prev and dXt are equal bit for bit;
dGs only re-associates and stays within the stack floor 1e-4 |ref| + 5e-5 mean|ref|.  Both are checked against the fp64
oracle as well."""
import pytest
import torch

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from stc_gnn_b200 import _lib
from tests.helpers import oracle_cell_with_grads, random_case
from tests.test_shared_terms_gpu import close, kinds_of_one_step, make_case, reference_rollout, run

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
FUSED, PAIR = 0, 1


def kinds_of(fn):
    fn()   # warm
    _lib.timing_enable(True)
    _lib.timing_collect()
    fn()
    torch.cuda.synchronize()
    _lib.timing_enable(False)
    return {k: v[1] for k, v in _lib.timing_collect().items()}


def cell_step(t, cfg, mode, preset):
    """One cell forward + backward with the given concurrency mode; Gs.grad starts from `preset` (None: no .grad)."""
    _lib.set_concurrency(mode)
    try:
        leaf = lambda x: x.float().to(DEV).requires_grad_(True)
        Gs, Gc, Xt, H, Wg, Wc, bg, bc = (leaf(t[k]) for k in ("Gs", "Gc", "Xt", "H", "Wg", "Wc", "bg", "bc"))
        if preset is not None:
            Gs.grad = preset.to(DEV).clone()

        def step():
            for p in (Gc, Xt, H, Wg, Wc, bg, bc):
                p.grad = None
            if preset is not None:
                Gs.grad.copy_(preset.to(DEV))
            else:
                Gs.grad = None
            Hn = S.stc_cell_forward(Gs, Gc, Xt, H, Wg, bg, Wc, bc, cfg["Ks"], cfg["Kc"])
            Hn.backward(t["dHn"].float().to(DEV))
            return Hn

        kinds = kinds_of(step)
        Hn = step()
        torch.cuda.synchronize()
        g = dict(dXt=Xt.grad, dH=H.grad, dWg=Wg.grad, dWc=Wc.grad, dGs=Gs.grad, dGc=Gc.grad, dbg=bg.grad, dbc=bc.grad)
        return Hn.detach().cpu(), {k: v.detach().cpu() for k, v in g.items()}, kinds
    finally:
        _lib.set_concurrency(-1)


# B, N, C, Din, h, Ks: hidden-side widths C*h = 16, 48, 80, 144 (48, 80 and 144 are not multiples of 32); x-side widths
# C*Din take the fused kernel too where they are multiples of 4.  B = 1, B < 148 SMs, several samples per CTA, and
# > 16 chunks per CTA (more than one dGs chain) at B = 600, W = 144.
CASES = [
    (3, 8, 1, 4, 16, 2),
    (2, 20, 3, 4, 16, 3),
    (1, 100, 5, 1, 16, 2),
    (300, 100, 5, 4, 16, 3),
    (600, 64, 9, 4, 16, 2),
    (40, 112, 3, 4, 16, 3),
]


@pytest.mark.parametrize("preset", [False, True])
@pytest.mark.parametrize("shape", CASES)
def test_fused_adjoint_matches_pair_and_oracle(shape, preset):
    B, N, C, Din, h, Ks = shape
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=2)
    t = random_case(B, N, C, Din, h, Ks, 2, seed=sum(shape))
    g0 = torch.randn(N, N, generator=torch.Generator().manual_seed(3)) * 0.1 if preset else None
    Hn_f, g_f, k_f = cell_step(t, cfg, FUSED, g0)
    Hn_p, g_p, k_p = cell_step(t, cfg, PAIR, g0)
    n_chains = (Ks - 1) * (2 + ((C * Din) % 4 == 0))   # d(rH), dH and (eligible width) dXt
    assert k_f.get("tc_support_adj") == n_chains and "tc_support_adj" not in k_p, (k_f, k_p)
    assert torch.equal(Hn_f, Hn_p)
    for k in ("dH", "dXt"):
        assert torch.equal(g_f[k], g_p[k]), f"{k} differs between the fused kernel and the pair"
    close(g_f["dGs"], g_p["dGs"], "dGs fused vs pair")
    Hn_o, g_o = oracle_cell_with_grads(t, cfg)
    if preset:
        g_o["dGs"] = g_o["dGs"] + g0.double()
    O.assert_close(Hn_f, Hn_o, "Hn")
    for k, v in g_f.items():
        O.assert_close(v, g_o[k], k)


def test_shared_terms_stack_with_fold():
    """Stack with shared hidden-state terms (a producer cell folds the adjoint of its reader), Ks = 3: the fused kernel
    runs every adjoint hop of the cells, and the result matches the pair and the unshared roll-out of independent cells."""
    case = make_case("dense", Ks=3, T=4, horizon=2, B=8)
    fn = lambda st, a, b, c: st(a, b, c)
    outs, kinds = {}, {}
    for mode in (FUSED, PAIR):
        _lib.set_concurrency(mode)
        try:
            kinds[mode] = kinds_of_one_step(fn, *case)
            outs[mode] = run(fn, *case)
        finally:
            _lib.set_concurrency(-1)
    # (Ks = 3: layer 0 is not hoisted, so every tc_outer of the pair is an adjoint step of a cell)
    assert kinds[FUSED].get("tc_support_adj", 0) > 0 and "tc_outer" not in kinds[FUSED], kinds
    assert kinds[FUSED]["tc_support_adj"] == kinds[PAIR]["tc_outer"] and "tc_support_adj" not in kinds[PAIR], kinds
    _lib.set_concurrency(FUSED)
    try:
        o_r, g_r = run(reference_rollout, *case)
    finally:
        _lib.set_concurrency(-1)
    (o_f, g_f), (o_p, g_p) = outs[FUSED], outs[PAIR]
    assert torch.equal(o_f, o_p) and torch.equal(o_f, o_r)
    for i, (a, b, r) in enumerate(zip(g_f, g_p, g_r)):
        close(a, b, f"grad {i} fused vs pair")
        close(a, r, f"grad {i} fused vs unshared roll-out")


def test_sf_launch_kinds_without_lanes():
    """SF stack at B = 1024 (side lanes inactive at the default concurrency): every adjoint hop of the cells is a
    tc_support_adj launch, tc_outer only runs the hoisted layer-0 product, tc_support only the forward hops."""
    case = make_case("dense", B=1024, T=4, horizon=2)
    fn = lambda st, a, b, c: st(a, b, c)
    got = kinds_of_one_step(fn, *case)
    _lib.set_concurrency(PAIR)
    try:
        pair = kinds_of_one_step(fn, *case)
    finally:
        _lib.set_concurrency(-1)
    assert got["tc_outer"] == 1, got
    assert got["tc_support_adj"] == pair["tc_outer"] - 1, (got, pair)
    assert got["tc_support"] + got["tc_support_adj"] == pair["tc_support"], (got, pair)
    for k in set(got) | set(pair):
        if k not in ("tc_support", "tc_outer", "tc_support_adj"):
            assert got.get(k) == pair.get(k), (k, got, pair)


@pytest.mark.parametrize("N", [113, 128])
def test_larger_supports_keep_the_pair(N):
    B, C, Din, h, Ks = 4, 5, 4, 16, 2
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=2)
    t = random_case(B, N, C, Din, h, Ks, 2, seed=N)
    Hn, g, kinds = cell_step(t, cfg, FUSED, None)
    assert "tc_support_adj" not in kinds and kinds.get("tc_outer") == 3, kinds
    Hn_o, g_o = oracle_cell_with_grads(t, cfg)
    O.assert_close(Hn, Hn_o, "Hn")
    O.assert_close(g["dGs"], g_o["dGs"], "dGs")
