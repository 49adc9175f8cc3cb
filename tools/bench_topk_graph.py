#!/usr/bin/env python
"""Cost of the sparse generator choosing its own pattern (`pair_topk` / stc_pair_topk, `SparseGraphGenerator(k=)`).

  config3  grid N = 4096, B = 8, T = 12, C = 16
  config4  kNN N = 65,536, B = 2, T = 12, C = 8

  python tools/bench_topk_graph.py [config3] [config4] [rows] > out.jsonl

For hg in {16, 64} (width W = B*T*hg) and k = 16 each line reports:
  - the selection kernel (CUDA events around many calls after a warm-up): ms, useful TFLOP/s from 2 N^2 (2W) (the 3xTF32
    tensor work is three times that), and its peak memory;
  - alternating with it in the same process, the obvious torch form of the same rule: row chunks of
    U_c V^T - V_c U^T, the diagonal set to 0, then torch.topk (ties are not ordered by column there), in fp32 (cuBLAS's
    default, the precision this project holds to) and with TF32 matmuls, each with its peak memory; the TF32 form's
    count of rows whose selected set differs from the kernel's, and the fp32 form's;
  - the generator's forward + backward with k = 16 against the same on the fixed pattern (grid / kNN).
`rows` (config 4, W = 384, k = 16): the selection of one rank's row block, n_rows = N / world for world 2, 4, 8
(`pair_topk(..., rows=)`, stc_pair_topk_rows), timed alternating with the full selection, with the segment count the
kernel chose for the block and whether the block is bitwise those rows of the full selection.
The first line names the device, its power limit and maximum SM clock.
"""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import stc_gnn_b200 as S  # noqa: E402
from stc_gnn_b200 import _lib  # noqa: E402
from stc_gnn_b200.synth import grid_csr, knn_csr  # noqa: E402

DEV = torch.device("cuda:0")
CONFIGS = {"config3": dict(N=4096, B=8, T=12, C=16), "config4": dict(N=65536, B=2, T=12, C=8)}
K = 16
ROUNDS = 5
CHUNK_BYTES = 4 << 30      # the torch form's [rows, N] score chunk (and its second product) stays under this


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


def alternate(variants, iters):
    for fn in variants.values():
        fn()
    torch.cuda.synchronize()
    out = {k: [] for k in variants}
    for _ in range(ROUNDS):
        for k, fn in variants.items():
            out[k].append(events_ms(fn, iters))
    return out


def summary(samples):
    return {"median": statistics.median(samples), "min": min(samples), "max": max(samples)}


def peak_bytes(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def torch_topk(U, V, k, tf32):
    """The chunked torch form: never more than CHUNK_BYTES of scores at once."""
    N = U.shape[0]
    rows = max(1, min(N, CHUNK_BYTES // (8 * N)))
    out = torch.empty(N, k, dtype=torch.int64, device=U.device)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    try:
        for r0 in range(0, N, rows):
            Sc = U[r0:r0 + rows] @ V.t()
            Sc.sub_(V[r0:r0 + rows] @ U.t())
            idx = torch.arange(r0, min(N, r0 + rows), device=U.device)
            Sc[idx - r0, idx] = 0
            out[r0:r0 + rows] = torch.topk(Sc, k, dim=1, sorted=False).indices
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return out


def rows_differing(a, b):
    return int((torch.sort(a.long(), 1).values != torch.sort(b.long(), 1).values).any(1).sum())


def bench(which, hg):
    cfg = CONFIGS[which]
    N, B, T, C = cfg["N"], cfg["B"], cfg["T"], cfg["C"]
    W = B * T * hg
    g = torch.Generator().manual_seed(hg)
    X = (torch.rand(B, T, N, C, generator=g) < 0.3).float().to(DEV)
    torch.manual_seed(hg)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    with torch.no_grad():
        Xn = X.permute(2, 0, 1, 3).reshape(N, B * T, C)
        U = torch.tanh(gen.alpha * (Xn @ gen.params_S["Wu"])).reshape(N, -1).contiguous()
        V = torch.tanh(gen.alpha * (Xn @ gen.params_S["Wv"])).reshape(N, -1).contiguous()
    flop = 2.0 * N * N * 2 * W
    iters = max(2, int(2e13 / flop))   # about a second of kernel time a round at 20 TFLOP/s
    variants = {"kernel": lambda: S.pair_topk(U, V, K),
                "torch_fp32": lambda: torch_topk(U, V, K, False),
                "torch_tf32": lambda: torch_topk(U, V, K, True)}
    t = alternate(variants, iters)
    mem = {name: peak_bytes(fn) for name, fn in variants.items()}
    sel = S.pair_topk(U, V, K)
    ms = statistics.median(t["kernel"])
    out = dict(kind="pair_topk", config=which, N=N, W=W, hg=hg, k=K, useful_flop=flop,
               kernel_ms=summary(t["kernel"]), kernel_useful_tflops=flop / ms / 1e9,
               kernel_tensor_tflops_3xtf32=3 * flop / ms / 1e9,
               torch_fp32_ms=summary(t["torch_fp32"]), torch_tf32_ms=summary(t["torch_tf32"]),
               speedup_vs_torch_fp32=statistics.median(t["torch_fp32"]) / ms,
               speedup_vs_torch_tf32=statistics.median(t["torch_tf32"]) / ms,
               rows_differing_torch_fp32=rows_differing(variants["torch_fp32"](), sel),
               rows_differing_torch_tf32=rows_differing(variants["torch_tf32"](), sel),
               peak_bytes=mem, workspace_bytes=_lib.load().stc_pair_topk_workspace_bytes(N, W, K),
               score_matrix_bytes=4 * N * N)
    # the generator's forward + backward, selected pattern against the fixed one
    r, c, v = grid_csr(64, 64) if which == "config3" else knn_csr(65536, 8)
    pat = S.CsrSupport(r.to(DEV), c.to(DEV), v.to(DEV), N)
    w_fixed, w_sel = torch.randn(pat.nnz, device=DEV), torch.randn(N * K, device=DEV)

    def step(k):
        gen.zero_grad(set_to_none=True)
        sup = gen(X, k=k) if k else gen(X, pat)
        (sup.vals * (w_sel if k else w_fixed)).sum().backward()

    gt = alternate({"selected_k16": lambda: step(K), "fixed_pattern": lambda: step(None)}, 10)
    out.update(generator_fwd_bwd_selected_ms=summary(gt["selected_k16"]),
               generator_fwd_bwd_fixed_ms=summary(gt["fixed_pattern"]), fixed_nnz=pat.nnz)
    emit(**out)


def bench_rows():
    N, W = 65536, 384
    U, V = (torch.tanh(torch.randn(N, W, generator=torch.Generator().manual_seed(s))).to(DEV) for s in (1, 2))
    lib = _lib.load()
    blocks = {w: (N // w, N // w) for w in (2, 4, 8)}     # rank 1's rows of an even split
    variants = {"full": lambda: S.pair_topk(U, V, K)}
    variants.update({f"world{w}": (lambda b=b: S.pair_topk(U, V, K, rows=b)) for w, b in blocks.items()})
    t = alternate(variants, 3)
    full = S.pair_topk(U, V, K)
    full_ms = statistics.median(t["full"])
    for w, (r0, n) in blocks.items():
        ws = lib.stc_pair_topk_rows_workspace_bytes(N, W, n, K)
        ms = statistics.median(t[f"world{w}"])
        emit(kind="pair_topk_rows", config="config4", N=N, W=W, k=K, world=w, row0=r0, n_rows=n,
             segments=ws // (8 * n * K), row_blocks=-(-n // 128), kernel_ms=summary(t[f"world{w}"]),
             full_selection_ms=summary(t["full"]), fraction_of_full=ms / full_ms, ideal_fraction=n / N,
             workspace_bytes=ws, full_workspace_bytes=lib.stc_pair_topk_workspace_bytes(N, W, K),
             bitwise_full_rows=bool(torch.equal(S.pair_topk(U, V, K, rows=(r0, n)), full[r0:r0 + n])))


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_topk_graph.py needs a CUDA device")
    _lib.load()
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the measurement still stands, but says that the limit is unknown
        smi = f"unavailable: {e!r}"
    emit(kind="device", name=torch.cuda.get_device_name(0), nvidia_smi=smi)
    for which in sys.argv[1:] or ["config3", "config4"]:
        if which == "rows":
            bench_rows()
            continue
        if which not in CONFIGS:
            raise SystemExit(f"unknown config {which!r} (use {', '.join(CONFIGS)})")
        for hg in (16, 64):
            bench(which, hg)


if __name__ == "__main__":
    main()
