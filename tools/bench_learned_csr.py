#!/usr/bin/env python
"""Cost of learnable edge values on a CSR spatial support (the edge gradient fused into the adjoint hop).

  hop      the adjoint hop alone: stc_support_apply_edge_grad vs the plain stc_support_apply (transpose = 0), at the
           shapes of bench_configs.py::bench_support (grid N = 4096, W = 1024, B = 16; kNN N = 65,536, W = 512, B = 2)
  config3  one cell training step (fwd + bwd), N = 4096 grid, C = 16, F = 64, Ks = Kc = 2, B = 8: constant vs learnable
  config4  one cell training step, N = 65,536 kNN, C = 8, F = 64, Ks = 4, Kc = 2, B = 2: constant vs learnable

  python tools/bench_learned_csr.py [hop] [config3] [config4] > out.jsonl

One JSON object per line.  The two variants of each comparison are timed in the same process, alternating, with CUDA
events around many launches; every operand is larger than the 126 MB L2 in the hop cases.  The first line names the
device, its power limit and maximum SM clock.
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

DEV = torch.device("cuda:0")
ROUNDS = 7


def emit(**kw):
    print(json.dumps(kw), flush=True)


def events_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def alternate(variants, iters, warm=3):
    """{name: [ms per call of each round]}: the variants take turns, ROUNDS times."""
    for fn in variants.values():
        for _ in range(warm):
            fn()
    torch.cuda.synchronize()
    out = {k: [] for k in variants}
    for _ in range(ROUNDS):
        for k, fn in variants.items():
            out[k].append(events_ms(fn, iters))
    return out


def summary(samples):
    return {"median": statistics.median(samples), "min": min(samples), "max": max(samples)}


def bench_hop():
    lib = _lib.load()
    r, c, v = grid_csr(64, 64)
    grid = S.CsrSupport(r.to(DEV), c.to(DEV), v.to(DEV), 4096)
    r, c, v = knn_csr(65536, 8)
    knn = S.CsrSupport(r.to(DEV), c.to(DEV), v.to(DEV), 65536)
    for name, sup, N, W, B in (("csr_grid_N4096_W1024", grid, 4096, 1024, 16), ("csr_knn_N65536_W512", knn, 65536, 512, 2)):
        X = torch.randn(B, N, W, device=DEV)
        A = torch.randn(B, N, W, device=DEV)
        Y = torch.empty_like(X)
        dvals = torch.zeros(sup.nnz, device=DEV)
        st, gs = torch.cuda.current_stream().cuda_stream, sup.struct()
        plain = lambda: lib.stc_support_apply(gs, N, B, W, 0, X.data_ptr(), N * W, None, N * W, Y.data_ptr(), 1.0, 0.0, st)
        fused = lambda: lib.stc_support_apply_edge_grad(gs, N, B, W, X.data_ptr(), N * W, None, N * W, Y.data_ptr(), 1.0,
                                                        0.0, A.data_ptr(), N * W, 1.0, dvals.data_ptr(), st)
        t = alternate({"plain": plain, "fused": fused}, iters=50)
        hop_bytes = 4.0 * B * N * W * 2 + 8.0 * sup.nnz + 4.0 * (N + 1)
        fused_bytes = hop_bytes + 4.0 * B * N * W + 4.0 * sup.nnz
        mp, mf = statistics.median(t["plain"]), statistics.median(t["fused"])
        emit(kind="hop", case=name, N=N, W=W, B=B, nnz=sup.nnz, plain_ms=summary(t["plain"]), fused_ms=summary(t["fused"]),
             plain_alg_bytes=hop_bytes, fused_alg_bytes=fused_bytes, plain_alg_GBs=hop_bytes / mp / 1e6,
             fused_alg_GBs=fused_bytes / mf / 1e6, ratio_fused_over_plain=mf / mp,
             operands_MB=4.0 * B * N * W * 3 / 1e6)
        del X, A, Y, dvals


def bench_cell(which):
    if which == "config3":
        N, C, F, B, Ks = 4096, 16, 64, 8, 2
        r, c, v = grid_csr(64, 64)
    else:
        N, C, F, B, Ks = 65536, 8, 64, 2, 4
        r, c, v = knn_csr(N, 8)
    const = S.CsrSupport(r.to(DEV), c.to(DEV), v.to(DEV), N)
    vals = torch.nn.Parameter(v.to(DEV).clone())
    learned = S.CsrSupport(r.to(DEV), c.to(DEV), vals, N)
    Gc = (torch.rand(C, C, generator=torch.Generator().manual_seed(0)) / C).to(DEV)
    torch.manual_seed(0)
    cell = S.STC_Cell(N, C, Ks, 2, F, F).to(DEV)
    X = torch.randn(B, N, C, F, device=DEV, requires_grad=True)
    H = (torch.randn(B, N, C, F, device=DEV) * 0.5).requires_grad_(True)
    dH = torch.randn(B, N, C, F, device=DEV)

    def step(sup):
        def run():
            for p in list(cell.parameters()) + [X, H, vals]:
                p.grad = None
            cell(Gs=sup, Gc=Gc, Xt=X, Ht_1=H).backward(dH)
        return run

    variants = {"constant": step(const), "learnable": step(learned)}
    t = alternate(variants, iters=10, warm=2)
    mc, ml = statistics.median(t["constant"]), statistics.median(t["learnable"])
    emit(kind=f"{which}_cell_train_step", N=N, C=C, F=F, B=B, Ks=Ks, Kc=2, nnz=const.nnz,
         constant_ms=summary(t["constant"]), learnable_ms=summary(t["learnable"]), ratio_learnable_over_constant=ml / mc,
         kernels_constant=kernel_breakdown(variants["constant"]), kernels_learnable=kernel_breakdown(variants["learnable"]))


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_learned_csr.py needs a CUDA device")
    _lib.load()
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the measurement still stands, but says that the limit is unknown
        smi = f"unavailable: {e!r}"
    emit(kind="device", name=torch.cuda.get_device_name(0), nvidia_smi=smi, rounds=ROUNDS)
    which = sys.argv[1:] or ["hop", "config3", "config4"]
    for w in which:
        {"hop": bench_hop, "config3": lambda: bench_cell("config3"), "config4": lambda: bench_cell("config4")}[w]()


if __name__ == "__main__":
    main()
