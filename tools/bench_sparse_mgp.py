#!/usr/bin/env python
"""Cost of the graph generator on a fixed CSR pattern (`SparseGraphGenerator`, stc_pair_scores_csr + stc_edge_softmax).

  config3  grid N = 4096, B = 8, T = 12, C = 16
  config4  kNN N = 65,536, B = 2, T = 12, C = 8; also the config 4 learnable cell training step (F = 64, Ks = 4, Kc = 2)
           with and without the generator in front of it, alternating in the same process

  python tools/bench_sparse_mgp.py [config3] [config4] > out.jsonl

For hg in {16, 64} (width = B*T*hg) each line reports: generator forward + backward ms with the kernel breakdown; the
scores kernel against the plain stc_support_apply hop on the same pattern at [1, N, 2*width] (the same neighbour
gathers), alternating; peak memory of the generator against the per-edge torch form (U[row], V[col], V[row], U[col]
gathered as [nnz, width] slabs); and parity_ok of P and the Wu / Wv gradients against that per-edge form evaluated in
fp64.  Timings are CUDA events around many calls after a warm-up.  The first line names the device, its power limit
and maximum SM clock.
"""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import stc_gnn_b200 as S  # noqa: E402
from stc_gnn_b200 import _lib  # noqa: E402
from stc_gnn_b200.synth import grid_csr, knn_csr  # noqa: E402
from bench_configs import kernel_breakdown  # noqa: E402
from bench_learned_csr import alternate, emit, events_ms, summary  # noqa: E402

DEV = torch.device("cuda:0")
CONFIGS = {"config3": dict(N=4096, B=8, T=12, C=16), "config4": dict(N=65536, B=2, T=12, C=8)}


def per_edge_generator(X, Wu, Wv, alpha, rows, col, N):
    """The obvious torch form: gathers four [nnz, width] endpoint slabs, kept by autograd for the backward."""
    B, T, _, C = X.shape
    U = torch.tanh(alpha * (X @ Wu)).permute(2, 0, 1, 3).reshape(N, -1)
    V = torch.tanh(alpha * (X @ Wv)).permute(2, 0, 1, 3).reshape(N, -1)
    Sc = (U[rows] * V[col]).sum(-1) - (V[rows] * U[col]).sum(-1)
    r = torch.relu(Sc)
    mx = torch.zeros(N, dtype=r.dtype, device=r.device).scatter_reduce(0, rows, r.detach(), "amax", include_self=True)
    ex = torch.exp(r - mx[rows])
    return ex / torch.zeros(N, dtype=r.dtype, device=r.device).index_add(0, rows, ex)[rows]


def max_err(got, ref, rtol, atol_scale):
    got, ref = got.double(), ref.double()
    scale = ref.abs().mean().item()
    err = (got - ref).abs()
    return int((err > rtol * ref.abs() + atol_scale * scale).sum().item()), err.max().item() / scale


def peak_bytes(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def pattern(which):
    r, c, v = grid_csr(64, 64) if which == "config3" else knn_csr(65536, 8)
    return S.CsrSupport(r.to(DEV), c.to(DEV), v.to(DEV), r.numel() - 1)


def bench_generator(which, pat, hg):
    cfg = CONFIGS[which]
    N, B, T, C = cfg["N"], cfg["B"], cfg["T"], cfg["C"]
    width = B * T * hg
    lib = _lib.load()
    g = torch.Generator().manual_seed(hg)
    X = (torch.rand(B, T, N, C, generator=g) < 0.3).float().to(DEV)
    torch.manual_seed(hg)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    w = torch.randn(pat.nnz, generator=g).to(DEV)

    def step():
        gen.zero_grad(set_to_none=False)
        (gen(X, pat).vals * w).sum().backward()

    step()
    torch.cuda.synchronize()
    gen_ms = alternate({"gen": step}, iters=20)["gen"]
    kernels = kernel_breakdown(step)
    gen_peak = peak_bytes(step)

    # scores kernel vs the plain hop with the same gathers ([1, N, 2 * width]; output slab written by the hop only)
    U = torch.randn(N, width, device=DEV)
    V = torch.randn(N, width, device=DEV)
    X2 = torch.randn(1, N, 2 * width, device=DEV)
    Y2 = torch.empty_like(X2)
    Sc = torch.empty(pat.nnz, device=DEV)
    st, gs = torch.cuda.current_stream().cuda_stream, pat.struct()
    scores = lambda: lib.stc_pair_scores_csr(gs, N, width, U.data_ptr(), V.data_ptr(), Sc.data_ptr(), st)
    hop = lambda: lib.stc_support_apply(gs, N, 1, 2 * width, 0, X2.data_ptr(), N * 2 * width, None, 0, Y2.data_ptr(),
                                        1.0, 0.0, st)
    t = alternate({"scores": scores, "hop": hop}, iters=50)
    ms_s, ms_h = statistics.median(t["scores"]), statistics.median(t["hop"])
    scores_bytes = 4.0 * 2 * N * width + 4.0 * 2 * width * pat.nnz + 8.0 * pat.nnz + 4.0 * (N + 1) + 4.0 * pat.nnz
    del U, V, X2, Y2, Sc

    # per-edge torch form: fp32 peak memory and time, fp64 for parity
    rows = torch.repeat_interleave(torch.arange(N, device=DEV), (pat.rowptr[1:] - pat.rowptr[:-1]).long())
    col = pat.col.long()
    Wu, Wv = gen.params_S["Wu"], gen.params_S["Wv"]
    out = dict(kind=f"{which}_generator", N=N, B=B, T=T, C=C, hg=hg, width=width, nnz=pat.nnz,
               gen_fwd_bwd_ms=summary(gen_ms), kernels=kernels, gen_peak_MB=gen_peak / 1e6,
               scores_ms=summary(t["scores"]), plain_hop_2w_ms=summary(t["hop"]), ratio_scores_over_hop=ms_s / ms_h,
               scores_alg_bytes=scores_bytes, scores_alg_GBs=scores_bytes / ms_s / 1e6,
               one_gathered_operand_MB=4.0 * pat.nnz * width / 1e6)
    try:
        a, b = Wu.detach().clone().requires_grad_(True), Wv.detach().clone().requires_grad_(True)

        def torch_step():
            a.grad = b.grad = None
            (per_edge_generator(X, a, b, gen.alpha, rows, col, N) * w).sum().backward()

        out["per_edge_torch_peak_MB"] = peak_bytes(torch_step) / 1e6
        torch_step()
        out["per_edge_torch_fwd_bwd_ms"] = events_ms(torch_step, 5)
        del a, b
    except torch.cuda.OutOfMemoryError:
        out["per_edge_torch_peak_MB"] = "out of memory"
    torch.cuda.empty_cache()
    step()
    a = Wu.detach().double().requires_grad_(True)
    b = Wv.detach().double().requires_grad_(True)
    P64 = per_edge_generator(X.double(), a, b, gen.alpha, rows, col, N)
    (P64 * w.double()).sum().backward()
    P = gen(X, pat).vals.detach()
    errs = dict(P=max_err(P, P64.detach(), 1e-4, 1e-5), dWu=max_err(Wu.grad, a.grad, 1e-4, 5e-5),
                dWv=max_err(Wv.grad, b.grad, 1e-4, 5e-5))
    out["parity_vs_fp64_per_edge"] = {k: {"n_outside": v[0], "worst_x_mean": v[1]} for k, v in errs.items()}
    out["parity_ok"] = all(v[0] == 0 for v in errs.values())
    del P64, a, b
    torch.cuda.empty_cache()
    emit(**out)


def bench_config4_step(pat):
    """One config 4 learnable cell training step, with the generator in front of it or on fixed learnable values."""
    N, C, F, B, Ks, T = 65536, 8, 64, 2, 4, 12
    g = torch.Generator().manual_seed(0)
    X_seq = (torch.rand(B, T, N, C, generator=g) < 0.3).float().to(DEV)
    Gc = (torch.rand(C, C, generator=g) / C).to(DEV)
    torch.manual_seed(0)
    cell = S.STC_Cell(N, C, Ks, 2, F, F).to(DEV)
    gen = S.SparseGraphGenerator(C, 16).to(DEV)
    with torch.no_grad():
        vals = torch.nn.Parameter(gen(X_seq, pat).vals.clone())
    fixed = pat.with_values(vals)
    X = torch.randn(B, N, C, F, device=DEV, requires_grad=True)
    H = (torch.randn(B, N, C, F, device=DEV) * 0.5).requires_grad_(True)
    dH = torch.randn(B, N, C, F, device=DEV)
    params = list(cell.parameters()) + list(gen.parameters()) + [X, H, vals]

    def run(with_gen):
        def f():
            for p in params:
                p.grad = None
            sup = gen(X_seq, pat) if with_gen else fixed
            cell(Gs=sup, Gc=Gc, Xt=X, Ht_1=H).backward(dH)
        return f

    variants = {"cell_step": run(False), "generator_plus_cell_step": run(True)}
    t = alternate(variants, iters=10, warm=2)
    mc, mg = statistics.median(t["cell_step"]), statistics.median(t["generator_plus_cell_step"])
    emit(kind="config4_learnable_cell_train_step", N=N, C=C, F=F, B=B, T=T, Ks=Ks, Kc=2, hg=16, nnz=pat.nnz,
         cell_step_ms=summary(t["cell_step"]), generator_plus_cell_step_ms=summary(t["generator_plus_cell_step"]),
         generator_share_of_one_cell_step=(mg - mc) / mg,
         kernels_generator_plus_cell_step=kernel_breakdown(variants["generator_plus_cell_step"]))


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse_mgp.py needs a CUDA device")
    _lib.load()
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the measurement still stands, but says that the limit is unknown
        smi = f"unavailable: {e!r}"
    emit(kind="device", name=torch.cuda.get_device_name(0), nvidia_smi=smi)
    for which in sys.argv[1:] or ["config3", "config4"]:
        pat = pattern(which)
        for hg in (16, 64):
            bench_generator(which, pat, hg)
        if which == "config4":
            bench_config4_step(pat)


if __name__ == "__main__":
    main()
