"""Forward-only cell calls (stc_cell_fwd_only: no backward state, no r / c / P_1 stores) against the training forward,
both under torch.no_grad.

Alternates cell.FORWARD_ONLY on and off in one process, `--rounds` rounds each, on
  sf_b512 / sf_b4096   the SF-shape RecurrentStack (N = 100, C = 5, h = 16, Din = 1, 2 layers, T = 9, horizon 3, dense Gs)
  g4096_b8             the grid-4096 stack (N = 4096, C = 16, h = 64, constant CSR support, encoder only, T = 12), B = 8
  config4_partitioned  one config 4 cell forward on a row-partitioned kNN support at world 1 (N = 65,536, C = 8,
                       Din = h = 64, Ks = 4), B = 2
and prints one JSON line per workload: the median milliseconds per call of each form and their ratio, the per-kernel
breakdown of one instrumented call per form (stc_timing_*: device ms, launches, algorithmic bytes), the peak memory a call
allocates beyond what was allocated before it, whether the two forms' outputs are bitwise equal, and the card name and
power limit read in the same process.  The SF inputs at B = 512 fit in L2; the others do not.
Usage: python tools/bench_forward_only.py [--rounds R] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import stc_gnn_b200 as S  # noqa: E402
from stc_gnn_b200 import _lib, cell  # noqa: E402

DEV = torch.device("cuda", 0)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # pragma: no cover
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unread ({e})"}


def stack_workload(N, C, h, Din, layers, T, horizon, B, csr):
    g = torch.Generator().manual_seed(0)
    torch.manual_seed(0)
    stack = S.RecurrentStack(N, C, 2, 2, Din, h, layers, horizon).to(DEV)
    if csr:   # constant 8-neighbour grid scaled by 1/8, as bench.py's g4096 workload
        from stc_gnn_b200.synth import grid_csr
        side = int(round(N ** 0.5))
        rp, ci, va = grid_csr(side, side)
        Gs = S.CsrSupport(rp.to(DEV), ci.to(DEV), va.to(DEV), N)
    else:     # the SF supports bench.py uses
        from stc_gnn_b200.synth import sf_supports
        Gs = sf_supports(seed=0)[0].to(DEV)
    Gc = (torch.rand(C, C, generator=g) * (2.0 / C)).to(DEV)
    X = (torch.rand(B, T, N, C, Din, generator=g) < 0.3).float().to(DEV)
    return lambda: stack(Gs, Gc, X)


def config4_workload(B=2):
    from stc_gnn_b200.halo import PartitionedSupport, partitioned_cell_forward
    from stc_gnn_b200.synth import knn_csr
    N, C, F, Ks, Kc = 65536, 8, 64, 4, 2
    rp, ci, va = knn_csr(N, 8)
    torch.manual_seed(0)
    c = S.STC_Cell(N, C, Ks, Kc, F, F).to(DEV)
    ps = PartitionedSupport(rp, ci, va, N, 0, 1)
    g = torch.Generator().manual_seed(100)
    Gc = (torch.rand(C, C, generator=g) / C).to(DEV)
    X = torch.randn(B, N, C, F, generator=g).to(DEV)
    H = (torch.randn(B, N, C, F, generator=g) * 0.5).to(DEV)
    return lambda: partitioned_cell_forward(ps, Gc, X, H, c.gates.W, c.gates.b, c.candi.W, c.candi.b, Ks, Kc)


WORKLOADS = {
    "sf_b512": lambda: stack_workload(100, 5, 16, 1, 2, 9, 3, 512, False),
    "sf_b4096": lambda: stack_workload(100, 5, 16, 1, 2, 9, 3, 4096, False),
    "g4096_b8": lambda: stack_workload(4096, 16, 64, 1, 2, 12, 0, 8, True),
    "config4_partitioned": config4_workload,
}


def timed(fn, iters):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / iters


def measure(name, make, rounds):
    fn = make()
    forms = {"forward_only": True, "training_forward": False}
    out, ms, peak, kinds = {}, {f: [] for f in forms}, {}, {}
    with torch.no_grad():
        for form, on in forms.items():   # warm both forms; the output of each
            cell.FORWARD_ONLY = on
            fn()
            out[form] = fn().clone()
        one = timed(fn, 1)
        iters = max(3, min(200, int(300.0 / max(one, 1e-3))))   # about 0.3 s of work per timed window
        for _ in range(rounds):
            for form, on in forms.items():
                cell.FORWARD_ONLY = on
                ms[form].append(timed(fn, iters))
        for form, on in forms.items():
            cell.FORWARD_ONLY = on
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            fn()
            torch.cuda.synchronize()
            peak[form] = torch.cuda.max_memory_allocated() - base
            _lib.timing_enable(True)
            _lib.timing_collect()
            fn()
            torch.cuda.synchronize()
            _lib.timing_enable(False)
            kinds[form] = {k: {"ms": round(v[0], 4), "launches": v[1], "alg_bytes": v[2]}
                           for k, v in _lib.timing_collect().items()}
    cell.FORWARD_ONLY = True
    med = {f: statistics.median(v) for f, v in ms.items()}
    return {"workload": name, "rounds": rounds, "iters_per_round": iters,
            "ms_per_call": {f: round(v, 4) for f, v in med.items()},
            "ms_per_call_all": {f: [round(x, 4) for x in v] for f, v in ms.items()},
            "ratio_forward_only_over_training": round(med["forward_only"] / med["training_forward"], 4),
            "peak_alloc_bytes": peak, "peak_ratio": round(peak["forward_only"] / max(peak["training_forward"], 1), 4),
            "bitwise_equal": bool(torch.equal(out["forward_only"], out["training_forward"])),
            "kinds": kinds, **card()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", nargs="*", default=None, help="workload names (default: all)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_forward_only.py measures on the GPU; no CUDA device is visible")
    _lib.load()
    lines = []
    for name, make in WORKLOADS.items():
        if args.only and name not in args.only:
            continue
        rec = measure(name, make, args.rounds)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
