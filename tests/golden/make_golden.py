"""Generate the golden vectors under tests/golden/ from the REAL reference.

Run in the build container only (needs /root/reference):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

The reference (pure PyTorch, /root/reference/framework/STC_GNN.py) is imported unmodified and
evaluated in fp64 (and fp32, for the record) on seeded inputs whose values are exactly
representable in fp32, so the GPU fp32 path and the fp64 oracle see identical inputs.
The reference has no tests or golden vectors of its own (SURVEY.md §4); these files are the pin.

Files written (all ``np.savez_compressed``):
  cell_<name>.npz   one STC_Cell forward + every gradient (STC_GNN.py:65-79 through autograd)
  stack_sf.npz      encoder(2 layers x T=9) + decoder(horizon 3) roll-out on real SF data with the
                    MGP_Gen-produced (denormal-laden) supports, outputs + gradients
  pred_sf.npz       the unmodified full STCGNN (STC_GNN.py:175-207; seeded init, Main.py's defaults) on the
                    FIRST TEST BATCH of the shipped SF split (Data_Container.py:56-66, 6:1:1, batch 32):
                    its own fp32 predictions, the supports its MGP_Gen produced, every cell / out_proj
                    weight, and the fp64 re-evaluation of encoder -> decoder -> out_proj -> sigmoid
  stack_longc.npz   BASELINE config 5 shapes (T = 48, C = 64 categories, h = 64, dense Gc): encoder + decoder
                    roll-out at B = 1 with every gradient; to stay small the fixture keeps the supports, the
                    outputs / input gradients of five nodes, every 4th row of each weight gradient, all bias and
                    support gradients, and checksums of the seeded inputs and weights the test regenerates
"""
import os
import sys

import numpy as np
import torch

REF = os.environ.get("STC_REF_DIR", "/root/reference/framework")
DATA = os.path.join(os.path.dirname(REF), "data", "SF-incidents-4h.npz")
OUT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF)
sys.dont_write_bytecode = True

import STC_GNN as ref  # noqa: E402


def f32exact(t):
    return t.float().double()


def gz(t):
    """gradient as numpy, zeros when autograd never touched the tensor (Ks=1 / Kc=1: support unused)."""
    return (t.grad if t.grad is not None else torch.zeros_like(t)).numpy()


def run_cell(name, B, N, C, Din, h, Ks, Kc, use_bias=True, act=None, seed=0, Gs=None, Gc=None, Xt=None,
             bias_scale=0.1, strided_T=None):
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    torch.set_default_dtype(torch.float64)
    activation = {None: None, "relu": torch.nn.ReLU}[act]
    cell = ref.STC_Cell(N, C, Ks, Kc, Din, h, use_bias=use_bias, activation=activation)
    with torch.no_grad():
        for p in cell.parameters():
            p.copy_(f32exact(p))
        if use_bias:
            cell.gates.b.copy_(f32exact(torch.randn(2 * h, generator=g) * bias_scale))
            cell.candi.b.copy_(f32exact(torch.randn(h, generator=g) * bias_scale))
    if Gs is None:
        Gs = torch.rand(N, N, generator=g) * (2.0 / N)
    if Gc is None:
        Gc = torch.rand(C, C, generator=g) * (2.0 / C)
    Gs = f32exact(Gs).requires_grad_(True)
    Gc = f32exact(Gc).requires_grad_(True)
    if Xt is None:
        if strided_T is not None:
            # the encoder hands the cell a [:, t] view whose batch stride is non-standard (STC_GNN.py:111)
            seq = f32exact(torch.randn(B, strided_T, N, C, Din, generator=g))
            Xt = seq[:, 1]
        else:
            Xt = f32exact(torch.randn(B, N, C, Din, generator=g))
    Xt = Xt.clone().requires_grad_(True)
    H = f32exact(torch.randn(B, N, C, h, generator=g) * 0.5).requires_grad_(True)
    dHn = f32exact(torch.randn(B, N, C, h, generator=g))

    Hn = cell(Gs=Gs, Gc=Gc, Xt=Xt, Ht_1=H)
    Hn.backward(dHn)
    out = dict(
        meta=np.array([B, N, C, Din, h, Ks, Kc, int(use_bias), 1 if act == "relu" else 0], dtype=np.int64),
        Gs=Gs.detach().float().numpy(), Gc=Gc.detach().float().numpy(),
        Xt=Xt.detach().float().numpy(), H=H.detach().float().numpy(), dHn=dHn.float().numpy(),
        Wg=cell.gates.W.detach().float().numpy(), Wc=cell.candi.W.detach().float().numpy(),
        Hn=Hn.detach().numpy(), dGs=gz(Gs), dGc=gz(Gc), dXt=Xt.grad.numpy(), dH=H.grad.numpy(),
        dWg=cell.gates.W.grad.numpy(), dWc=cell.candi.W.grad.numpy(),
    )
    if use_bias:
        out.update(bg=cell.gates.b.detach().float().numpy(), bc=cell.candi.b.detach().float().numpy(),
                   dbg=cell.gates.b.grad.numpy(), dbc=cell.candi.b.grad.numpy())
    # the reference evaluated in its native fp32, for the record (noise floor of the reference itself)
    torch.set_default_dtype(torch.float32)
    cell32 = ref.STC_Cell(N, C, Ks, Kc, Din, h, use_bias=use_bias, activation=activation)
    cell32.load_state_dict({k: v.float() for k, v in cell.state_dict().items()})
    Hn32 = cell32(Gs=Gs.detach().float(), Gc=Gc.detach().float(), Xt=Xt.detach().float(), Ht_1=H.detach().float())
    out["Hn_ref_fp32"] = Hn32.detach().numpy()
    np.savez_compressed(os.path.join(OUT, f"cell_{name}.npz"), **out)
    print(f"cell_{name}: |Hn|={Hn.abs().mean():.4f} fp32-vs-fp64 max {np.abs(out['Hn_ref_fp32'] - out['Hn']).max():.2e}")


def sf_supports_and_data(B=2):
    """Real SF data slice and the supports the real MGP_Gen produces from it (denormal-laden Gs)."""
    d = np.load(DATA)
    inc = torch.from_numpy(d["incident"].reshape(d["incident"].shape[0], 100, 5).astype(np.float32))
    As = torch.from_numpy(d["s_adj"]).float()
    Ac = torch.from_numpy(d["c_cor"]).float()
    T = 9
    # supports come from a full training batch of 32 windows (Data_Container.py:107-112), as in a real
    # forward: the batch/time-summed scores (STC_GNN.py:231-232) are large enough that the softmax
    # underflows into zeros and fp32 denormals; only B windows are kept as cell inputs.
    X32 = torch.stack([inc[i:i + T] for i in range(32)], dim=0)             # [32,T,N,C]
    torch.set_default_dtype(torch.float32)
    torch.manual_seed(0)
    mgp = ref.MGP_Gen(100, 5, 16)
    with torch.no_grad():
        Gs, Gc = mgp(X32, As, Ac)
    return X32[:B].clone(), Gs.detach(), Gc.detach()


def run_stack(X_seq, Gs, Gc):
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(1)
    N, C, h, Ks, Kc, layers, horizon = 100, 5, 16, 2, 2, 2, 3
    enc = ref.STC_Encoder(N, C, Ks, Kc, 1, h, layers)
    dec = ref.STC_Decoder(N, C, Ks, Kc, h, h, layers, horizon)
    with torch.no_grad():
        for p in list(enc.parameters()) + list(dec.parameters()):
            p.copy_(f32exact(p))
    Gs = f32exact(Gs).requires_grad_(True)
    Gc = f32exact(Gc).requires_grad_(True)
    X = f32exact(X_seq).unsqueeze(-1).requires_grad_(True)
    _, Ht = enc(Gs=Gs, Gc=Gc, X_seq=X, H0_l=None)
    inp = Ht[-1]
    outs = []
    for _ in range(horizon):
        Hl, Ht = dec(Gs=Gs, Gc=Gc, Xt=inp, H0_l=Ht)
        inp = Hl
        outs.append(Hl)
    out = torch.stack(outs, dim=1)
    g = torch.Generator().manual_seed(2)
    dOut = f32exact(torch.randn(out.shape, generator=g))
    out.backward(dOut)
    save = dict(meta=np.array([X.shape[0], 9, N, C, 1, h, Ks, Kc, layers, horizon], dtype=np.int64),
                X_seq=X.detach().float().numpy(), Gs=Gs.detach().float().numpy(), Gc=Gc.detach().float().numpy(),
                dOut=dOut.float().numpy(), out=out.detach().numpy(), dGs=Gs.grad.numpy(), dGc=Gc.grad.numpy(),
                dX_seq=X.grad.numpy())
    for tag, mod in (("enc", enc), ("dec", dec)):
        for i, cell in enumerate(mod.cell_list):
            for conv in ("gates", "candi"):
                for pn in ("W", "b"):
                    p = getattr(getattr(cell, conv), pn)
                    save[f"{tag}{i}_{conv}_{pn}"] = p.detach().float().numpy()
                    save[f"d_{tag}{i}_{conv}_{pn}"] = p.grad.numpy()
    np.savez_compressed(os.path.join(OUT, "stack_sf.npz"), **save)
    den = ((Gs.detach().float().abs() < 1.1754944e-38) & (Gs.detach() != 0)).float().mean().item()
    print(f"stack_sf: out mean|.|={out.abs().mean():.4f}; Gs denormal fraction {den:.3f}, "
          f"zero fraction {(Gs.detach() == 0).float().mean():.3f}")


def run_predictions():
    """BASELINE.json north_star: 'predictions on the shipped SF-incidents-4h data must match'."""
    import Data_Container as dc   # the reference's own windowing and split
    d = np.load(DATA)
    gen = dc.DataGenerator(obs_len=9, pred_len=3, data_split_ratio=(6, 1, 1))
    loaders = gen.get_data_loader(params=dict(H=10, W=10, C=5, device="cpu", batch_size=32), data=dict(inc=d["incident"]))
    X, Y = next(iter(loaders["test"]))                                   # [32,9,100,5], [32,3,100,5]
    As = torch.from_numpy(d["s_adj"]).float()
    Ac = torch.from_numpy(d["c_cor"]).float()
    torch.set_default_dtype(torch.float32)
    torch.manual_seed(0)
    model = ref.STCGNN(100, 5, 2, 2, 1, 16, 2, 3)                        # Model_Trainer.py:39-46 with Main.py defaults
    model.eval()
    with torch.no_grad():
        pred32 = model(X, As, Ac)                                        # the reference's own answer, fp32
        Gs, Gc = model.mix_graph_pair(X, As, Ac)
    # fp64 re-evaluation of everything after MGP_Gen, from the fp32 supports and weights
    torch.set_default_dtype(torch.float64)
    enc = ref.STC_Encoder(100, 5, 2, 2, 1, 16, 2, return_all_layers=True)
    dec = ref.STC_Decoder(100, 5, 2, 2, 16, 16, 2, 3)
    enc.load_state_dict({k: v.double() for k, v in model.encoder.state_dict().items()})
    dec.load_state_dict({k: v.double() for k, v in model.decoder.state_dict().items()})
    W1, b1 = model.out_proj[0].weight.double(), model.out_proj[0].bias.double()
    W2, b2 = model.out_proj[1].weight.double(), model.out_proj[1].bias.double()
    with torch.no_grad():
        Gs64, Gc64 = Gs.double(), Gc.double()
        _, Ht = enc(Gs=Gs64, Gc=Gc64, X_seq=X.double().unsqueeze(-1), H0_l=None)
        inp, outs = Ht[-1], []
        for _ in range(3):
            Hl, Ht = dec(Gs=Gs64, Gc=Gc64, Xt=inp, H0_l=Ht)
            inp = Hl
            outs.append(Hl)
        hid = torch.stack(outs, dim=1)
        pred64 = torch.sigmoid((hid @ W1.t() + b1) @ W2.t() + b2).squeeze(-1)
    save = dict(meta=np.array([32, 9, 100, 5, 1, 16, 2, 2, 2, 3], dtype=np.int64),
                X_seq=X.numpy().astype(np.uint8), Y=Y.numpy().astype(np.uint8), Gs=Gs.numpy(), Gc=Gc.numpy(),
                pred=pred64.numpy(), pred_ref_fp32=pred32.numpy(),
                out_W1=W1.detach().float().numpy(), out_b1=b1.detach().float().numpy(),
                out_W2=W2.detach().float().numpy(), out_b2=b2.detach().float().numpy())
    for tag, mod in (("enc", model.encoder), ("dec", model.decoder)):
        for i, cell in enumerate(mod.cell_list):
            for conv in ("gates", "candi"):
                for pn in ("W", "b"):
                    save[f"{tag}{i}_{conv}_{pn}"] = getattr(getattr(cell, conv), pn).detach().float().numpy()
    np.savez_compressed(os.path.join(OUT, "pred_sf.npz"), **save)
    print(f"pred_sf: predictions in [{pred64.min():.3f}, {pred64.max():.3f}]; reference fp32 vs fp64 max-abs "
          f"{(pred32.double() - pred64).abs().max():.2e}, max-rel {((pred32.double() - pred64).abs() / pred64.abs()).max():.2e}")


LONGC = dict(B=1, T=48, N=100, C=64, Din=1, h=64, Ks=2, Kc=2, layers=2, horizon=3)
LONGC_NODES = [0, 7, 33, 50, 99]          # output / input-gradient rows kept in the fixture
LONGC_ROW_STEP = 4                        # every 4th row of each weight gradient is kept
LONGC_DROP_BITS = 16                      # low mantissa bits rounded off the fp64 arrays: keeps the file under 1 MB


def round_mantissa(a, bits=LONGC_DROP_BITS):
    """fp64 array rounded to nearest with its `bits` low mantissa bits zero (relative change <= 2^(bits-53), 7.3e-12
    for 16: far inside the rtol 1e-9 the oracle is held to); zlib then compresses those bytes away."""
    if a.dtype != np.float64 or a.ndim == 0:
        return a
    u = a.view(np.uint64)
    return ((u + np.uint64(1 << (bits - 1))) & ~np.uint64((1 << bits) - 1)).view(np.float64)


def longc_inputs():
    """Seeded inputs of the BASELINE config 5 roll-out (T = 48, C = 64 categories, dense learned-like Gc), shared by
    this generator and tests/test_cell_gpu.py::test_config5_longc_rollout (the fixture stores only their checksums).
    Imports nothing from the product package: the same recipe is restated in tests/helpers.py::longc_case."""
    c = LONGC
    g = torch.Generator().manual_seed(48)
    X = (torch.rand(c["B"], c["T"], c["N"], c["C"], 1, generator=g) < 0.1635).float()
    N, C = c["N"], c["C"]
    Ps = torch.softmax(torch.relu(torch.randn(N, N, generator=g) * 3.0), dim=-1)
    Gs = (0.5 * Ps + 0.5 * torch.rand(N, N, generator=g) * (2.0 / N)).float()
    Gc = (0.5 * torch.softmax(torch.relu(torch.randn(C, C, generator=g) * 3.0), dim=-1)
          + 0.5 * torch.rand(C, C, generator=g) * (2.0 / C)).float()
    dOut = torch.randn(c["B"], c["horizon"], N, C, c["h"], generator=g).float()
    return X, Gs, Gc, dOut


def run_longc():
    """BASELINE config 5 shapes: the reference's encoder (2 layers x T = 48) + decoder (horizon 3) at C = 64, h = 64."""
    c = LONGC
    X, Gs, Gc, dOut = longc_inputs()
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(5)
    enc = ref.STC_Encoder(c["N"], c["C"], c["Ks"], c["Kc"], c["Din"], c["h"], c["layers"])
    dec = ref.STC_Decoder(c["N"], c["C"], c["Ks"], c["Kc"], c["h"], c["h"], c["layers"], c["horizon"])
    with torch.no_grad():
        for p in list(enc.parameters()) + list(dec.parameters()):
            p.copy_(f32exact(p))
    Gs64 = Gs.double().requires_grad_(True)
    Gc64 = Gc.double().requires_grad_(True)
    X64 = X.double().requires_grad_(True)
    _, Ht = enc(Gs=Gs64, Gc=Gc64, X_seq=X64, H0_l=None)
    inp, outs = Ht[-1], []
    for _ in range(c["horizon"]):
        Hl, Ht = dec(Gs=Gs64, Gc=Gc64, Xt=inp, H0_l=Ht)
        inp = Hl
        outs.append(Hl)
    out = torch.stack(outs, dim=1)
    out.backward(dOut.double())
    save = dict(meta=np.array([c[k] for k in ("B", "T", "N", "C", "Din", "h", "Ks", "Kc", "layers", "horizon")], dtype=np.int64),
                nodes=np.array(LONGC_NODES), row_step=np.array(LONGC_ROW_STEP), weight_seed=np.array(5),
                Gs=Gs.numpy(), Gc=Gc.numpy(), X_bits=np.packbits(X.numpy().astype(np.uint8)),
                dOut_checksum=np.array(dOut.double().abs().sum().item()),
                out_nodes=out.detach()[:, :, LONGC_NODES].numpy(), out_abs_mean=np.array(out.detach().abs().mean().item()),
                dGs=Gs64.grad.numpy(), dGc=Gc64.grad.numpy(), dX_nodes=X64.grad[:, :, LONGC_NODES].numpy(),
                dX_abs_mean=np.array(X64.grad.abs().mean().item()))
    wsum = 0.0
    for tag, mod in (("enc", enc), ("dec", dec)):
        for i, cell in enumerate(mod.cell_list):
            for conv in ("gates", "candi"):
                W, b = getattr(cell, conv).W, getattr(cell, conv).b
                wsum += W.detach().abs().sum().item()
                save[f"d_{tag}{i}_{conv}_W_rows"] = W.grad[::LONGC_ROW_STEP].float().numpy()
                save[f"d_{tag}{i}_{conv}_W_abs_mean"] = np.array(W.grad.abs().mean().item())
                save[f"d_{tag}{i}_{conv}_b"] = b.grad.numpy()
    save["weight_checksum"] = np.array(wsum)
    np.savez_compressed(os.path.join(OUT, "stack_longc.npz"), **{k: round_mantissa(v) for k, v in save.items()})
    print(f"stack_longc: out mean|.|={out.abs().mean():.4f}, dGc mean|.|={Gc64.grad.abs().mean():.3e}, "
          f"weights |.|_1={wsum:.6f}")


if __name__ == "__main__":
    if "--longc-only" in sys.argv:
        run_longc()
        sys.exit(0)
    if "--pred-only" in sys.argv:
        run_predictions()
        sys.exit(0)
    run_cell("tiny", B=2, N=7, C=3, Din=1, h=4, Ks=2, Kc=2, seed=1)
    run_cell("k33", B=2, N=9, C=4, Din=3, h=5, Ks=3, Kc=3, seed=2)
    run_cell("k42_relu", B=1, N=8, C=2, Din=2, h=4, Ks=4, Kc=2, act="relu", seed=3)
    run_cell("k24_nobias", B=3, N=5, C=6, Din=2, h=3, Ks=2, Kc=4, use_bias=False, seed=4)
    run_cell("k11", B=2, N=6, C=3, Din=2, h=4, Ks=1, Kc=1, seed=5)
    run_cell("strided", B=3, N=10, C=5, Din=1, h=8, Ks=2, Kc=2, seed=6, strided_T=4)
    X_seq, Gs, Gc = sf_supports_and_data(B=2)
    run_cell("sf_din1", B=2, N=100, C=5, Din=1, h=16, Ks=2, Kc=2, seed=7, Gs=Gs, Gc=Gc,
             Xt=f32exact(X_seq[:, 3]).unsqueeze(-1))
    run_cell("sf_din16", B=2, N=100, C=5, Din=16, h=16, Ks=2, Kc=2, seed=8, Gs=Gs, Gc=Gc)
    run_stack(X_seq, Gs, Gc)
    run_predictions()
    run_longc()
