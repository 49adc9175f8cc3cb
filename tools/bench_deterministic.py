"""Cost of the deterministic mode (torch.use_deterministic_algorithms(True): fixed-order gradient reductions).

Alternates the default and the deterministic mode in one process, `--rounds` rounds each, on
  sf_b4096 / sf_b512 / sf_b32   the SF-shape RecurrentStack (N = 100, C = 5, h = 16, dense learnable Gs), one training step
  sf_b32_graph                  the same at B = 32 as a GraphedStep replay (captured once per mode)
  g4096_b8                      the grid-4096 stack (N = 4096, C = 16, h = 64, CSR support), B = 8
  config4_cell                  one learnable-CSR cell step at N = 65,536, B = 2 (C = 8, Din = h = 64, Ks = 4)
and prints one JSON line per workload: median step time per mode and their ratio, the deterministic step once more with
torch.utils.deterministic.fill_uninitialized_memory = False (the cost of torch's NaN fill of fresh buffers), the per-kernel breakdown of one
instrumented step per mode (a run of its own), whether two runs of each mode gave bitwise-equal gradients, and the card
name and power limit read in the same process.  Usage: python tools/bench_deterministic.py [--out FILE]
"""
import argparse
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

DEV = torch.device("cuda", 0)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # pragma: no cover
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unread ({e})"}


def stack_workload(N, C, h, Din, Ks, Kc, layers, T, horizon, B, csr):
    g = torch.Generator().manual_seed(0)
    stack = S.RecurrentStack(N, C, Ks, Kc, Din, h, layers, horizon).to(DEV)
    if csr:   # constant 8-neighbour grid scaled by 1/8, as bench.py's g4096 workload
        from stc_gnn_b200.synth import grid_csr
        side = int(round(N ** 0.5))
        rp, ci, va = grid_csr(side, side)
        Gs = S.CsrSupport(rp.to(DEV), ci.to(DEV), va.to(DEV), N)
        leaves = []
    else:     # the SF supports bench.py uses, Gs learnable
        from stc_gnn_b200.synth import sf_supports
        Gs = sf_supports(seed=0)[0].to(DEV).requires_grad_(True)
        leaves = [Gs]
    Gc = (torch.rand(C, C, generator=g) * (2.0 / C)).to(DEV).requires_grad_(True)
    X = torch.randn(B, T, N, C, Din, generator=g).to(DEV)
    params = list(stack.parameters()) + leaves + [Gc]

    def step():
        for p in params:
            p.grad = None
        out = stack(Gs, Gc, X)
        out.square().mean().backward()
        return [p.grad for p in params]
    return step


def graphed_workload():
    """SF stack at B = 32 as a CUDA-graph replay; one graph per mode, captured on the mode's first call."""
    graphs = {}
    g = torch.Generator().manual_seed(0)
    from stc_gnn_b200.synth import sf_supports
    stack = S.RecurrentStack(100, 5, 2, 2, 1, 16, 2, 3).to(DEV)
    Gs = sf_supports(seed=0)[0].to(DEV).requires_grad_(True)
    Gc = (torch.rand(5, 5, generator=g) * 0.4).to(DEV).requires_grad_(True)
    X = torch.randn(32, 9, 100, 5, 1, generator=g).to(DEV)
    params = list(stack.parameters()) + [Gs, Gc]
    loss_fn = lambda Xs: stack(Gs, Gc, Xs).square().mean()

    def step():
        mode = torch.are_deterministic_algorithms_enabled()
        if mode not in graphs:
            graphs[mode] = S.GraphedStep(loss_fn, [X], params)
        graphs[mode].replay(X)
        return [p.grad for p in params]
    return step


def config4_workload():
    N, C, Din, h, Ks, Kc, B, deg = 65536, 8, 64, 64, 4, 2, 2, 8
    g = torch.Generator().manual_seed(0)
    cols = torch.stack([torch.randperm(N, generator=g)[:deg] for _ in range(64)])   # 64 distinct rows of columns,
    cols = cols.repeat(N // 64, 1)                                                  # tiled over all N rows
    cols, _ = cols.sort(dim=1)
    rowptr = torch.arange(0, N * deg + 1, deg, dtype=torch.int32)
    vals = torch.nn.Parameter((torch.rand(N * deg, generator=g) * (1.0 / deg)).to(DEV))
    sup = S.CsrSupport(rowptr.to(DEV), cols.reshape(-1).int().to(DEV), vals, N)
    cell = S.STC_Cell(N, C, Ks, Kc, Din, h).to(DEV)
    Xt = torch.randn(B, N, C, Din, generator=g).to(DEV)
    H = torch.randn(B, N, C, h, generator=g).to(DEV)
    Gc = (torch.rand(C, C, generator=g) * (2.0 / C)).to(DEV).requires_grad_(True)
    params = list(cell.parameters()) + [vals, Gc]

    def step():
        for p in params:
            p.grad = None
        cell(sup, Gc, Xt, H).square().mean().backward()
        return [p.grad for p in params]
    return step


def time_steps(step, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def breakdown(step):
    _lib.timing_enable(True)
    _lib.timing_collect()
    step()
    torch.cuda.synchronize()
    _lib.timing_enable(False)
    return {k: {"ms": round(v[0], 4), "launches": v[1]} for k, v in sorted(_lib.timing_collect().items())}


def bitwise_repeat(step):
    a = [x.detach().clone() for x in step() if x is not None]
    b = [x.detach().clone() for x in step() if x is not None]
    torch.cuda.synchronize()
    return all(torch.equal(x, y) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    args = ap.parse_args()
    info = card()
    SF = dict(N=100, C=5, h=16, Din=1, Ks=2, Kc=2, layers=2, T=9, horizon=3, csr=False)
    G4 = dict(N=4096, C=16, h=64, Din=1, Ks=2, Kc=2, layers=2, T=12, horizon=0, csr=True)
    workloads = {
        "sf_b4096": lambda: stack_workload(B=4096, **SF),
        "sf_b512": lambda: stack_workload(B=512, **SF),
        "sf_b32": lambda: stack_workload(B=32, **SF),
        "sf_b32_graph": graphed_workload,
        "g4096_b8": lambda: stack_workload(B=8, **G4),
        "config4_cell": config4_workload,
    }
    if args.only:
        workloads = {k: v for k, v in workloads.items() if k in args.only.split(",")}
    lines = []
    for name, make in workloads.items():
        step = make()
        times = {"default": [], "deterministic": []}
        for _ in range(args.rounds):
            for mode in ("default", "deterministic"):
                torch.use_deterministic_algorithms(mode == "deterministic")
                step()
                step()
                times[mode].append(time_steps(step, args.steps))
        rec = {"workload": name, **info, "rounds": args.rounds, "steps_per_round": args.steps}
        for mode in ("default", "deterministic"):
            torch.use_deterministic_algorithms(mode == "deterministic")
            rec[f"step_ms_{mode}"] = round(statistics.median(times[mode]), 3)
            rec[f"step_ms_{mode}_all"] = [round(t, 3) for t in times[mode]]
            rec[f"kernel_breakdown_{mode}"] = breakdown(step)
            rec[f"bitwise_repeat_{mode}"] = bitwise_repeat(step)
        rec["ratio_deterministic_over_default"] = round(rec["step_ms_deterministic"] / rec["step_ms_default"], 4)
        if name != "sf_b32_graph":   # (a replay allocates nothing: no fill to switch off)
            import torch.utils.deterministic as D
            torch.use_deterministic_algorithms(True)
            D.fill_uninitialized_memory = False
            step()
            nofill = [time_steps(step, args.steps) for _ in range(args.rounds)]
            D.fill_uninitialized_memory = True
            rec["step_ms_deterministic_no_nan_fill"] = round(statistics.median(nofill), 3)
            rec["nan_fill_ms"] = round(rec["step_ms_deterministic"] - rec["step_ms_deterministic_no_nan_fill"], 3)
        torch.use_deterministic_algorithms(False)
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)
        del step
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
