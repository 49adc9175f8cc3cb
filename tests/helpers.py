"""Shared test helpers: golden loading and seeded case construction."""
import glob
import os

import numpy as np
import torch

from oracle import stc_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CELL_CASES = sorted(os.path.basename(p)[5:-4] for p in glob.glob(os.path.join(GOLDEN, "cell_*.npz")))
GRAD_KEYS = ("dXt", "dH", "dWg", "dWc", "dbg", "dbc", "dGs", "dGc")


def load_cell(name):
    z = np.load(os.path.join(GOLDEN, f"cell_{name}.npz"))
    B, N, C, Din, h, Ks, Kc, use_bias, relu = (int(v) for v in z["meta"])
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, use_bias=bool(use_bias), activation="relu" if relu else None)
    t = {k: torch.from_numpy(z[k]) for k in z.files if k != "meta"}
    return cfg, t


def load_stack():
    z = np.load(os.path.join(GOLDEN, "stack_sf.npz"))
    B, T, N, C, Din, h, Ks, Kc, layers, horizon = (int(v) for v in z["meta"])
    cfg = dict(B=B, T=T, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, layers=layers, horizon=horizon)
    t = {k: torch.from_numpy(z[k]) for k in z.files if k != "meta"}
    return cfg, t


def load_pred():
    """Full-model predictions of the unmodified reference on the first SF test batch (tests/golden/make_golden.py)."""
    z = np.load(os.path.join(GOLDEN, "pred_sf.npz"))
    B, T, N, C, Din, h, Ks, Kc, layers, horizon = (int(v) for v in z["meta"])
    cfg = dict(B=B, T=T, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, layers=layers, horizon=horizon)
    t = {k: torch.from_numpy(z[k]) for k in z.files if k != "meta"}
    t["X_seq"] = t["X_seq"].float().unsqueeze(-1)      # stored as uint8 incident flags [B,T,N,C]
    return cfg, t


def random_case(B, N, C, Din, h, Ks, Kc, seed=0, use_bias=True, sparse_frac=None, dtype=torch.float64):
    """Seeded inputs with fp32-exact values. ``sparse_frac`` zeroes that fraction of Gs (for CSR tests)."""
    g = torch.Generator().manual_seed(seed)
    f = lambda t: t.float().to(dtype)
    Gs = torch.rand(N, N, generator=g) * (2.0 / max(N, 1))
    if sparse_frac is not None:
        Gs = Gs * (torch.rand(N, N, generator=g) >= sparse_frac) * (1.0 / max(1e-3, 1.0 - sparse_frac))
    Gc = torch.rand(C, C, generator=g) * (2.0 / C)
    p = O.xavier_cell_params(Din, h, Ks, Kc, g, dtype=torch.float32, use_bias=use_bias, bias_scale=0.1)
    case = dict(Gs=f(Gs), Gc=f(Gc), Xt=f(torch.randn(B, N, C, Din, generator=g)),
                H=f(torch.randn(B, N, C, h, generator=g) * 0.5), dHn=f(torch.randn(B, N, C, h, generator=g)),
                Wg=f(p.Wg), Wc=f(p.Wc), bg=f(p.bg) if use_bias else None, bc=f(p.bc) if use_bias else None)
    return case


def oracle_cell_with_grads(t, cfg, dtype=torch.float64):
    """Run the lean oracle through autograd; returns (Hn, grads dict)."""
    names = ["Gs", "Gc", "Xt", "H", "Wg", "Wc"] + (["bg", "bc"] if t.get("bg") is not None else [])
    v = {}
    for k in names:
        x = t[k]
        x = x.to_dense() if x.layout != torch.strided else x
        v[k] = x.to(dtype).clone().requires_grad_(True)
    Hn = O.stc_cell(v["Gs"], v["Gc"], v["Xt"], v["H"], v["Wg"], v.get("bg"), v["Wc"], v.get("bc"),
                    cfg["Ks"], cfg["Kc"], cfg.get("activation"))
    Hn.backward(t["dHn"].to(dtype))
    z = lambda k: v[k].grad if v[k].grad is not None else torch.zeros_like(v[k])
    grads = dict(dXt=z("Xt"), dH=z("H"), dWg=z("Wg"), dWc=z("Wc"), dGs=z("Gs"), dGc=z("Gc"))
    if "bg" in v:
        grads.update(dbg=z("bg"), dbc=z("bc"))
    return Hn.detach(), grads


def find_reference():
    """Directory holding the UNMODIFIED reference's framework/*.py, or None.  The reference is not part of this
    repository: point $STC_REF_DIR at a checkout's framework/ directory, or stage one under baseline/_ref
    (tools/stage_reference.sh).  Tests that need the live reference skip when this returns None."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for cand in (os.environ.get("STC_REF_DIR"), os.path.join(root, "baseline", "_ref", "framework")):
        if cand and os.path.isfile(os.path.join(cand, "STC_GNN.py")):
            return cand
    return None


def import_reference():
    """Import the reference's STC_GNN module (unmodified) from find_reference(); returns (module, framework_dir)."""
    import importlib
    import sys
    ref = find_reference()
    if ref is None:
        return None, None
    sys.dont_write_bytecode = True
    if ref not in sys.path:
        sys.path.insert(0, ref)
    return importlib.import_module("STC_GNN"), ref


def longc_case():
    """BASELINE config 5 roll-out fixture (tests/golden/stack_longc.npz, written by make_golden.py::run_longc from the
    imported reference).  The seeded inputs and weights are regenerated here -- same recipe as make_golden.py::
    longc_inputs -- and verified against the checksums the fixture stores.  Returns (cfg, tensors, golden npz)."""
    z = np.load(os.path.join(GOLDEN, "stack_longc.npz"))
    B, T, N, C, Din, h, Ks, Kc, layers, horizon = (int(v) for v in z["meta"])
    cfg = dict(B=B, T=T, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, layers=layers, horizon=horizon)
    g = torch.Generator().manual_seed(48)
    X = (torch.rand(B, T, N, C, 1, generator=g) < 0.1635).float()
    Ps = torch.softmax(torch.relu(torch.randn(N, N, generator=g) * 3.0), dim=-1)
    Gs = (0.5 * Ps + 0.5 * torch.rand(N, N, generator=g) * (2.0 / N)).float()
    Gc = (0.5 * torch.softmax(torch.relu(torch.randn(C, C, generator=g) * 3.0), dim=-1)
          + 0.5 * torch.rand(C, C, generator=g) * (2.0 / C)).float()
    dOut = torch.randn(B, horizon, N, C, h, generator=g).float()
    assert np.array_equal(np.packbits(X.numpy().astype(np.uint8)), z["X_bits"]), "seeded X differs from the fixture's"
    assert np.array_equal(Gs.numpy(), z["Gs"]) and np.array_equal(Gc.numpy(), z["Gc"]), "seeded supports differ"
    assert abs(dOut.double().abs().sum().item() - float(z["dOut_checksum"])) < 1e-6 * float(z["dOut_checksum"])
    # weights: the reference's construction order and init (encoder cells then decoder cells, gates.W before candi.W,
    # xavier-normal W / zero b, STC_GNN.py:17-21,57-58,95,151) under torch.manual_seed(weight_seed) in fp64, rounded to fp32
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(int(z["weight_seed"]))
        cells = []
        for i in range(2 * layers):
            din = Din if i == 0 else h
            Wg = torch.nn.init.xavier_normal_(torch.empty((din + h) * Ks * Kc, 2 * h))
            Wc = torch.nn.init.xavier_normal_(torch.empty((din + h) * Ks * Kc, h))
            cells.append(O.CellParams(Wg.float().double(), torch.zeros(2 * h, dtype=torch.float64), Wc.float().double(),
                                      torch.zeros(h, dtype=torch.float64)))
    finally:
        torch.set_default_dtype(prev)
    wsum = sum(float(p.Wg.abs().sum() + p.Wc.abs().sum()) for p in cells)
    assert abs(wsum - float(z["weight_checksum"])) < 1e-9 * wsum, (wsum, float(z["weight_checksum"]))
    return cfg, dict(X=X, Gs=Gs, Gc=Gc, dOut=dOut, enc=cells[:layers], dec=cells[layers:]), z
