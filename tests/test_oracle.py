"""CPU tests: the oracle (oracle/stc_oracle.py) against the golden vectors generated from the real
reference (tests/golden/make_golden.py), against its own analytic backward, and -- when the reference
tree is present (build container only) -- against the live reference."""
import sys

import pytest
import torch

from oracle import stc_oracle as O
from tests.helpers import (CELL_CASES, GRAD_KEYS, find_reference, load_cell, load_pred, load_stack, oracle_cell_with_grads,
                           random_case)

REF_DIR = find_reference()


def test_golden_files_present():
    assert len(CELL_CASES) >= 8, CELL_CASES


@pytest.mark.parametrize("name", CELL_CASES)
def test_oracle_matches_golden_cell(name):
    cfg, t = load_cell(name)
    Hn, grads = oracle_cell_with_grads(t, cfg)
    # fp64 vs fp64: only summation order differs -> 1e-9 relative
    O.assert_close(Hn, t["Hn"], f"{name}:Hn", rtol=1e-9, atol_scale=1e-10)
    for k in GRAD_KEYS:
        if k in t:
            O.assert_close(grads[k], t[k], f"{name}:{k}", rtol=1e-9, atol_scale=1e-9)


@pytest.mark.parametrize("name", CELL_CASES)
def test_analytic_backward_matches_golden(name):
    cfg, t = load_cell(name)
    d = lambda k: t[k].double() if k in t else None
    g = O.stc_cell_backward(d("Gs"), d("Gc"), d("Xt"), d("H"), d("Wg"), d("bg"), d("Wc"), d("bc"),
                            cfg["Ks"], cfg["Kc"], d("dHn"), cfg["activation"])
    for k in GRAD_KEYS:
        if k in t:
            O.assert_close(g[k], t[k], f"{name}:{k}", rtol=1e-9, atol_scale=1e-9)


@pytest.mark.parametrize("name", ["tiny", "k33", "sf_din16"])
def test_refshape_matches_lean(name):
    cfg, t = load_cell(name)
    d = lambda k: t[k].double() if k in t else None
    a = O.stc_cell_refshape(d("Gs"), d("Gc"), d("Xt"), d("H"), d("Wg"), d("bg"), d("Wc"), d("bc"),
                            cfg["Ks"], cfg["Kc"], cfg["activation"])
    O.assert_close(a, t["Hn"], name, rtol=1e-9, atol_scale=1e-10)


def test_reference_fp32_noise_floor_is_inside_tolerance():
    """The tolerance must at least admit the reference's own fp32 evaluation."""
    for name in CELL_CASES:
        _, t = load_cell(name)
        O.assert_close(t["Hn_ref_fp32"], t["Hn"], name)


def test_sparse_support_equals_dense():
    cfg = dict(B=2, N=40, C=3, Din=2, h=4, Ks=4, Kc=2)
    t = random_case(**cfg, seed=11, sparse_frac=0.8)
    a = O.stc_cell(t["Gs"], t["Gc"], t["Xt"], t["H"], t["Wg"], t["bg"], t["Wc"], t["bc"], 4, 2)
    b = O.stc_cell(t["Gs"].to_sparse_csr(), t["Gc"], t["Xt"], t["H"], t["Wg"], t["bg"], t["Wc"], t["bc"], 4, 2)
    O.assert_close(b, a, "csr", rtol=1e-12, atol_scale=1e-12)
    g1 = O.stc_cell_backward(t["Gs"], t["Gc"], t["Xt"], t["H"], t["Wg"], t["bg"], t["Wc"], t["bc"], 4, 2, t["dHn"])
    g2 = O.stc_cell_backward(t["Gs"].to_sparse_csr(), t["Gc"], t["Xt"], t["H"], t["Wg"], t["bg"], t["Wc"],
                             t["bc"], 4, 2, t["dHn"])
    for k in ("dXt", "dH", "dWg", "dWc", "dGc"):
        O.assert_close(g2[k], g1[k], k, rtol=1e-11, atol_scale=1e-11)
    assert g2["dGs"] is None


def test_stack_matches_golden():
    cfg, t = load_stack()
    enc, dec, leaves = [], [], {}
    for tag, lst in (("enc", enc), ("dec", dec)):
        for i in range(cfg["layers"]):
            ps = []
            for conv in ("gates", "candi"):
                for pn in ("W", "b"):
                    k = f"{tag}{i}_{conv}_{pn}"
                    leaves[k] = t[k].double().requires_grad_(True)
                    ps.append(leaves[k])
            lst.append(O.CellParams(*ps))
    Gs = t["Gs"].double().requires_grad_(True)
    Gc = t["Gc"].double().requires_grad_(True)
    X = t["X_seq"].double().requires_grad_(True)
    out = O.stack_forward(Gs, Gc, X, enc, dec, cfg["horizon"], cfg["Ks"], cfg["Kc"])
    O.assert_close(out, t["out"], "stack out", rtol=1e-9, atol_scale=1e-10)
    out.backward(t["dOut"].double())
    O.assert_close(Gs.grad, t["dGs"], "dGs", rtol=1e-8, atol_scale=1e-9)
    O.assert_close(Gc.grad, t["dGc"], "dGc", rtol=1e-8, atol_scale=1e-9)
    O.assert_close(X.grad, t["dX_seq"], "dX_seq", rtol=1e-8, atol_scale=1e-9)
    for k, v in leaves.items():
        O.assert_close(v.grad, t["d_" + k], k, rtol=1e-8, atol_scale=1e-9)


def test_predictions_on_shipped_sf_test_batch_match_golden():
    """Encoder -> decoder -> out_proj -> sigmoid (STC_GNN.py:191-207) on the first SF test batch, fp64 oracle vs the
    fp64 evaluation of the reference's own modules; the reference's native fp32 answer must sit inside rtol 1e-4."""
    cfg, t = load_pred()
    enc, dec = [], []
    for tag, lst in (("enc", enc), ("dec", dec)):
        for i in range(cfg["layers"]):
            lst.append(O.CellParams(*[t[f"{tag}{i}_{conv}_{pn}"].double() for conv in ("gates", "candi") for pn in ("W", "b")]))
    hid = O.stack_forward(t["Gs"].double(), t["Gc"].double(), t["X_seq"].double(), enc, dec, cfg["horizon"], cfg["Ks"], cfg["Kc"])
    pred = torch.sigmoid((hid @ t["out_W1"].double().t() + t["out_b1"].double()) @ t["out_W2"].double().t()
                         + t["out_b2"].double()).squeeze(-1)
    assert pred.shape == t["pred"].shape == (32, 3, 100, 5)
    O.assert_close(pred, t["pred"], "SF predictions", rtol=1e-9, atol_scale=0.0)
    O.assert_close(t["pred_ref_fp32"], t["pred"], "reference fp32 predictions", rtol=1e-4, atol_scale=0.0)


def test_grid_adjacency_matches_shipped_shape():
    A = O.grid_adjacency(10, 10)
    assert int(A.sum()) == 684 and bool((A == A.t()).all()) and float(A.diagonal().abs().sum()) == 0.0
    assert sorted(set(A.sum(1).tolist())) == [3.0, 5.0, 8.0]


@pytest.mark.skipif(REF_DIR is None, reason="needs the live reference (set STC_REF_DIR)")
@pytest.mark.parametrize("Ks,Kc,act", [(2, 2, None), (3, 2, "relu"), (4, 3, None)])
def test_oracle_matches_live_reference(Ks, Kc, act):
    sys.dont_write_bytecode = True
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import STC_GNN as ref
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        cfg = dict(B=2, N=11, C=4, Din=3, h=6, Ks=Ks, Kc=Kc)
        t = random_case(**cfg, seed=Ks * 10 + Kc)
        cell = ref.STC_Cell(11, 4, Ks, Kc, 3, 6, activation=torch.nn.ReLU if act else None)
        with torch.no_grad():
            cell.gates.W.copy_(t["Wg"]); cell.gates.b.copy_(t["bg"])
            cell.candi.W.copy_(t["Wc"]); cell.candi.b.copy_(t["bc"])
        leaves = {k: t[k].clone().requires_grad_(True) for k in ("Gs", "Gc", "Xt", "H")}
        Hn = cell(Gs=leaves["Gs"], Gc=leaves["Gc"], Xt=leaves["Xt"], Ht_1=leaves["H"])
        Hn.backward(t["dHn"])
        cfg["activation"] = act
        Hn_o, g = oracle_cell_with_grads(t, cfg)
        O.assert_close(Hn_o, Hn.detach(), "Hn", rtol=1e-10, atol_scale=1e-11)
        O.assert_close(g["dGs"], leaves["Gs"].grad, "dGs", rtol=1e-9, atol_scale=1e-9)
        O.assert_close(g["dGc"], leaves["Gc"].grad, "dGc", rtol=1e-9, atol_scale=1e-9)
        O.assert_close(g["dXt"], leaves["Xt"].grad, "dXt", rtol=1e-9, atol_scale=1e-9)
        O.assert_close(g["dH"], leaves["H"].grad, "dH", rtol=1e-9, atol_scale=1e-9)
        O.assert_close(g["dWg"], cell.gates.W.grad, "dWg", rtol=1e-9, atol_scale=1e-9)
        O.assert_close(g["dbc"], cell.candi.b.grad, "dbc", rtol=1e-9, atol_scale=1e-9)
    finally:
        torch.set_default_dtype(old)


def test_oracle_matches_reference_longc_rollout():
    """BASELINE config 5 shapes (T = 48, C = 64, h = 64): oracle roll-out and gradients vs the reference's fixture."""
    from tests.helpers import longc_case
    cfg, t, z = longc_case()
    Gs = t["Gs"].double().requires_grad_(True)
    Gc = t["Gc"].double().requires_grad_(True)
    X = t["X"].double().requires_grad_(True)
    cells = t["enc"] + t["dec"]
    for p in cells:
        for w in p.tensors():
            w.requires_grad_(True)
    out = O.stack_forward(Gs, Gc, X, t["enc"], t["dec"], cfg["horizon"], cfg["Ks"], cfg["Kc"])
    out.backward(t["dOut"].double())
    nodes, step = list(z["nodes"]), int(z["row_step"])
    O.assert_close(out.detach()[:, :, nodes], torch.from_numpy(z["out_nodes"]), "longc out", 1e-9, 1e-10)
    O.assert_close(Gs.grad, torch.from_numpy(z["dGs"]), "longc dGs", 1e-8, 1e-9)
    O.assert_close(Gc.grad, torch.from_numpy(z["dGc"]), "longc dGc", 1e-8, 1e-9)
    O.assert_close(X.grad[:, :, nodes], torch.from_numpy(z["dX_nodes"]), "longc dX", 1e-8, 1e-9)
    for name, p in zip(("enc0", "enc1", "dec0", "dec1"), cells):
        for conv, W, b in (("gates", p.Wg, p.bg), ("candi", p.Wc, p.bc)):
            O.assert_close(W.grad[::step], torch.from_numpy(z[f"d_{name}_{conv}_W_rows"]).double(), f"longc d{name}.{conv}.W",
                           1e-6, 1e-7)     # the fixture keeps these rows in fp32
            O.assert_close(b.grad, torch.from_numpy(z[f"d_{name}_{conv}_b"]), f"longc d{name}.{conv}.b", 1e-8, 1e-9)


def test_subgraph_closure_reproduces_full_problem_gradients():
    """The property tests/test_cell_gpu.py::test_config4_knn65536_f64_forward_backward_exact_subgraph relies on: with the
    output gradient confined to a node block S, the cell restricted to the 2(Ks-1)-hop closure U of S has the same
    H'[S], parameter / Gc gradients and (dXt, dH)[U] as the full graph, and the full gradients vanish outside U."""
    import numpy as np
    import scipy.sparse as sp
    from stc_gnn_b200.synth import knn_csr
    from tests.helpers import oracle_cell_with_grads
    N, C, Din, h, Ks, Kc, B = 2048, 2, 3, 4, 4, 2, 2
    rp, ci, va = knn_csr(N, 8, 1)
    A = sp.csr_matrix((va.numpy().astype(np.float64), ci.numpy(), rp.numpy()), shape=(N, N))
    struct = ((abs(A) + abs(A).T) > 0).astype(np.float32)
    lo, hi = 700, 732
    m = np.zeros(N, np.float32)
    m[lo:hi] = 1
    for _ in range(2 * (Ks - 1)):
        m = ((struct @ m + m) > 0).astype(np.float32)
    U = np.nonzero(m)[0]
    assert U.size < N // 2
    g = torch.Generator().manual_seed(1)
    p = O.xavier_cell_params(Din, h, Ks, Kc, g, dtype=torch.float64, bias_scale=0.1)
    t = dict(Gc=torch.rand(C, C, generator=g, dtype=torch.float64) / C, Xt=torch.randn(B, N, C, Din, generator=g, dtype=torch.float64),
             H=torch.randn(B, N, C, h, generator=g, dtype=torch.float64), Wg=p.Wg, Wc=p.Wc, bg=p.bg, bc=p.bc)
    t["dHn"] = torch.zeros(B, N, C, h, dtype=torch.float64)
    t["dHn"][:, lo:hi] = torch.randn(B, hi - lo, C, h, generator=g, dtype=torch.float64)
    coo = A.tocoo()
    t["Gs"] = torch.sparse_coo_tensor(np.stack([coo.row, coo.col]), torch.from_numpy(coo.data), size=(N, N)).coalesce()
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, activation=None)
    Hn_f, g_f = oracle_cell_with_grads(t, cfg)
    sub = A[U][:, U].tocoo()
    Ut = torch.from_numpy(U)
    ts = dict(t, Gs=torch.sparse_coo_tensor(np.stack([sub.row, sub.col]), torch.from_numpy(sub.data), size=(U.size, U.size)).coalesce(),
              Xt=t["Xt"][:, Ut], H=t["H"][:, Ut], dHn=t["dHn"][:, Ut])
    Hn_s, g_s = oracle_cell_with_grads(ts, dict(cfg, N=int(U.size)))
    pos = np.searchsorted(U, np.arange(lo, hi))
    O.assert_close(Hn_s[:, pos], Hn_f[:, lo:hi], "H'[S]", 1e-12, 1e-13)
    for k in ("dWg", "dWc", "dbg", "dbc", "dGc"):
        O.assert_close(g_s[k], g_f[k], k, 1e-11, 1e-12)
    outside = torch.ones(N, dtype=torch.bool)
    outside[Ut] = False
    for k in ("dXt", "dH"):
        O.assert_close(g_s[k], g_f[k][:, Ut], k, 1e-11, 1e-12)
        assert float(g_f[k][:, outside].abs().max()) == 0.0
