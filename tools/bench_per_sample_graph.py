#!/usr/bin/env python
"""Cost of per-sample spatial graphs (a CsrSupport with values [B, nnz]) against one graph shared by the batch.

  hop      the forward hop alone (stc_support_apply, transpose = 1), shared values vs per-sample values, at the shapes of
           bench_learned_csr.py (grid N = 4096, W = 1024, B = 16; kNN N = 65,536, W = 512, B = 2), in GB/s of
           algorithmic bytes (per-sample: + 4 (B - 1) nnz bytes of values)
  config3  one cell training step (fwd + bwd), N = 4096 grid, C = 16, F = 64, Ks = Kc = 2, B = 8: shared learnable
           values [nnz] vs per-sample learnable values [B, nnz]
  config4  the same on N = 65,536 kNN, C = 8, F = 64, Ks = 4, Kc = 2, B = 2
  gen3 / gen4  the sparse graph generator, forward + backward, hg = 16, T = 12, on the config 3 / config 4 pattern:
           batch-summed (P [nnz]) vs per sample (P [B, nnz])

  python tools/bench_per_sample_graph.py [hop] [config3] [config4] [gen3] [gen4] > out.jsonl

One JSON object per line; the two variants of each comparison alternate in the same process (medians of 7 rounds, CUDA
events around many calls).  The hop operands are larger than the 126 MB L2.  The first line names the device, its power
limit and maximum SM clock, read in the same process.
"""
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
from bench_learned_csr import alternate, emit, summary  # noqa: E402

DEV = torch.device("cuda:0")


def pattern(which):
    if which == "config3":
        return 4096, grid_csr(64, 64)
    return 65536, knn_csr(65536, 8)


def bench_hop():
    lib = _lib.load()
    for name, which, W, B in (("csr_grid_N4096_W1024", "config3", 1024, 16), ("csr_knn_N65536_W512", "config4", 512, 2)):
        N, (r, c, v) = pattern(which)
        shared = S.CsrSupport(r.to(DEV), c.to(DEV), v.to(DEV).requires_grad_(True), N)
        per = S.CsrSupport(r.to(DEV), c.to(DEV), v.to(DEV)[None].repeat(B, 1), N)
        X = torch.randn(B, N, W, device=DEV)
        Y = torch.empty_like(X)
        st = torch.cuda.current_stream().cuda_stream
        g1, g2 = shared.struct(), per.struct()
        hop = lambda gs: (lambda: lib.stc_support_apply(gs, N, B, W, 1, X.data_ptr(), N * W, None, N * W, Y.data_ptr(),
                                                        1.0, 0.0, st))
        t = alternate({"shared": hop(g1), "per_sample": hop(g2)}, iters=50)
        nnz = shared.nnz
        b_shared = 4.0 * B * N * W * 2 + 8.0 * nnz + 4.0 * (N + 1)
        b_per = b_shared + 4.0 * (B - 1) * nnz
        ms, mp = statistics.median(t["shared"]), statistics.median(t["per_sample"])
        emit(kind="hop", case=name, N=N, W=W, B=B, nnz=nnz, shared_ms=summary(t["shared"]),
             per_sample_ms=summary(t["per_sample"]), shared_alg_bytes=b_shared, per_sample_alg_bytes=b_per,
             shared_alg_GBs=b_shared / ms / 1e6, per_sample_alg_GBs=b_per / mp / 1e6,
             ratio_per_sample_over_shared=mp / ms, operands_MB=4.0 * B * N * W * 2 / 1e6)
        del X, Y


def bench_cell(which):
    N, (r, c, v) = pattern(which)
    C, F, Ks, B = (16, 64, 2, 8) if which == "config3" else (8, 64, 4, 2)
    vs = torch.nn.Parameter(v.to(DEV).clone())
    vp = torch.nn.Parameter(v.to(DEV)[None].repeat(B, 1).contiguous())
    shared = S.CsrSupport(r.to(DEV), c.to(DEV), vs, N)
    per = S.CsrSupport(r.to(DEV), c.to(DEV), vp, N)
    Gc = (torch.rand(C, C, generator=torch.Generator().manual_seed(0)) / C).to(DEV)
    torch.manual_seed(0)
    cell = S.STC_Cell(N, C, Ks, 2, F, F).to(DEV)
    X = torch.randn(B, N, C, F, device=DEV, requires_grad=True)
    H = (torch.randn(B, N, C, F, device=DEV) * 0.5).requires_grad_(True)
    dH = torch.randn(B, N, C, F, device=DEV)

    def step(sup):
        def run():
            for p in list(cell.parameters()) + [X, H, vs, vp]:
                p.grad = None
            cell(Gs=sup, Gc=Gc, Xt=X, Ht_1=H).backward(dH)
        return run

    variants = {"shared": step(shared), "per_sample": step(per)}
    t = alternate(variants, iters=10, warm=2)
    ms, mp = statistics.median(t["shared"]), statistics.median(t["per_sample"])
    emit(kind=f"{which}_cell_train_step", N=N, C=C, F=F, B=B, Ks=Ks, Kc=2, nnz=shared.nnz,
         shared_learnable_ms=summary(t["shared"]), per_sample_learnable_ms=summary(t["per_sample"]),
         ratio_per_sample_over_shared=mp / ms, kernels_shared=kernel_breakdown(variants["shared"]),
         kernels_per_sample=kernel_breakdown(variants["per_sample"]))


def bench_gen(which):
    N, (r, c, v) = pattern("config3" if which == "gen3" else "config4")
    C, B = (16, 8) if which == "gen3" else (8, 2)
    T, hg = 12, 16
    pat = S.CsrSupport(r.to(DEV), c.to(DEV), v.to(DEV), N)
    torch.manual_seed(0)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    X = torch.randn(B, T, N, C, device=DEV)
    dP1 = torch.randn(pat.nnz, device=DEV)
    dPB = torch.randn(B, pat.nnz, device=DEV)

    def run(per_sample):
        def go():
            for p in gen.parameters():
                p.grad = None
            P = gen(X, pat, per_sample=per_sample).vals
            (P * (dPB if per_sample else dP1)).sum().backward()
        return go

    t = alternate({"batch_summed": run(False), "per_sample": run(True)}, iters=10, warm=2)
    mb, mp = statistics.median(t["batch_summed"]), statistics.median(t["per_sample"])
    emit(kind=f"{which}_generator_fwd_bwd", N=N, C=C, B=B, T=T, hg=hg, nnz=pat.nnz,
         batch_summed_ms=summary(t["batch_summed"]), per_sample_ms=summary(t["per_sample"]),
         ratio_per_sample_over_batch_summed=mp / mb)


def main():
    which = sys.argv[1:] or ["hop", "config3", "config4", "gen3", "gen4"]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    emit(kind="device", name=torch.cuda.get_device_name(0), nvidia_smi=smi)
    for w in which:
        if w == "hop":
            bench_hop()
        elif w.startswith("config"):
            bench_cell(w)
        else:
            bench_gen(w)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
