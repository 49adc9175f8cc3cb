#!/usr/bin/env python
"""bench.py -- train samples/s (forward+backward) of the STC-GNN recurrent cell stack on B200.

Workload (BASELINE.json configs[1], "synthetic SF-shape tensors ... on 1xB200"): the SF-shape
recurrent stack -- encoder 2 layers x T=9 + decoder horizon 3 x 2 layers = 24 cell steps per sample
(N=100 regions, C=5 categories, h=16, Ks=Kc=2, dense learned-like Gs requiring grad), i.e. the
reference's STCGNN.forward/backward minus MGP_Gen and out_proj -- the hot path this repo replaces.
One "step" = forward + backward of one batch of B windows per GPU; a sample = one [T,N,C] window.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference] [--dump-outputs DIR]

`--dump-outputs DIR` also writes what the last timed step computed (loss, stack output, every gradient) as
DIR/<name>.npy, so that two builds can be compared output for output.

Prints ONE JSON line (rank 0).  `value` = device-resident throughput; `e2e` = the same through the
public module API with host (pinned) inputs copied in and the loss read back every step;
`roofline` = the dominant kernel's algorithmic bytes / its device time (CUDA events around every launch
of that kernel during a second, instrumented pass over the same K steps) against the measured HBM peak;
`roofline_step` = the whole step against SURVEY 8d's fused-cell floor (ALG_BYTES_TRAIN); `cpu_baseline` = the
reference's cell stack on this box's host cores on a bounded sample -- the UNMODIFIED reference when the probe finds
it ($STC_REF_DIR, /root/reference/framework, baseline/_ref/framework; kind "reference"), else the oracle's
reference-shaped port (kind "port") -- default and flush-denormal; `gpu_eager_baseline` = the same stack run by stock
PyTorch eager on this GPU (the kernels to beat), swept over B in {32, 512, 4096} next to this repo's own numbers.
`--impl reference` runs only the CPU arm (rank 0) and prints the same line shape.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from

import numpy as np  # noqa: E402
import torch  # noqa: E402

SF = dict(N=100, C=5, h=16, Din=1, Ks=2, Kc=2, layers=2, T=9, horizon=3, grid=(10, 10))
# BASELINE.json configs[2] (side workload, --workload g4096): 64x64 grid, constant CSR support, encoder only
G4096 = dict(N=4096, C=16, h=64, Din=1, Ks=2, Kc=2, layers=2, T=12, horizon=0, grid=(64, 64))
WL = SF          # selected in main() from --workload
METRIC = "train samples/s (fwd+bwd), SF-shape STC cell stack"
UNIT = "samples/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--batch", type=int, default=4096, help="windows per GPU per step (weak scaling)")
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--cpu-batch", type=int, default=128, help="windows per CPU-baseline step (bounded sample)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-eager-baseline", action="store_true", help="skip the stock-PyTorch-eager-on-GPU sweep")
    p.add_argument("--no-roofline", action="store_true", help="skip the instrumented per-kernel pass")
    p.add_argument("--workload", default="sf", choices=["sf", "g4096"],
                   help="sf = BASELINE configs[1] (headline); g4096 = configs[2]: N=4096 grid, C=16, F=64, T=12, CSR support "
                        "(default batch 4 per GPU; no CPU arm)")
    p.add_argument("--cuda-graph", action="store_true",
                   help="capture the whole fwd+bwd step once and replay it (stc_gnn_b200.GraphedStep; N=1 only)")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write the last timed step's loss, stack output (a fixed sample of it above 4 M elements) and "
                        "gradients as DIR/<name>.npy")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def measured_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed ncu --set full capture
    (profiles/traffic.json, written by tools/profile_summary.py traffic); None when that kernel was not captured."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None, None
    with open(path) as f:
        d = json.load(f)
    e = d.get("kernels", {}).get(kernel)
    if not e:
        return None, None
    return e["dram_bytes_per_launch"], f"{d.get('source', 'profiles/traffic.json')}: mean of {e['launches']} captured launches at batch {d.get('batch')}"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# synthetic SF-shape inputs (SURVEY.md §8d config 2)
# ------------------------------------------------------------------------------------------------
def synthetic_inputs(B, seed, device="cpu", pin=False):
    from stc_gnn_b200.synth import sf_supports
    g = torch.Generator().manual_seed(seed)
    X = (torch.rand(B, WL["T"], WL["N"], WL["C"], 1, generator=g) < 0.1635).float()   # Bernoulli(data mean)
    y = (torch.rand(B, WL["horizon"] or WL["T"], WL["N"], WL["C"], generator=g) < 0.1635).float()
    if WL is SF:
        Gs, Gc = sf_supports(seed=0)
    else:   # constant supports: the CSR grid is built on the device by the caller, Gc ~ U(0,1)/C (SURVEY 8d config 3)
        Gs, Gc = None, torch.rand(WL["C"], WL["C"], generator=torch.Generator().manual_seed(0)) / WL["C"]
    if pin:
        X, y = X.pin_memory(), y.pin_memory()
    return X, y, Gs, Gc


def loss_fn(out, y):
    """Stand-in for out_proj + loss: mean over the hidden axis, squared error against the target."""
    return (out.mean(dim=-1) - y).square().mean()


DUMP_SAMPLE = 4 << 20      # elements kept of an output larger than this (16 MB of fp32)
DUMP_LIMIT = 64 << 20      # bytes written by --dump-outputs in all


def dump_outputs(path, arrays):
    """Write {name: tensor} as path/<name>.npy in float32.  A tensor of more than DUMP_SAMPLE elements is replaced by
    the elements at DUMP_SAMPLE positions drawn (with a fixed seed, sorted) from its flattened index range: the same
    positions on every run with the same arguments."""
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        a = t.float().cpu().numpy()
        total += a.nbytes
        if total > DUMP_LIMIT:
            raise SystemExit(f"--dump-outputs: more than {DUMP_LIMIT} bytes")
        np.save(os.path.join(path, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc, self.path = None, f"/tmp/stc_clocks_{os.getpid()}.csv"
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "power_w_max": max(power), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# The reference's cell stack through stock PyTorch: the CPU arm (cpu_baseline / --impl reference) and the
# eager-on-GPU arm.  The UNMODIFIED reference is used when the probe finds it; else the oracle's reference-shaped port.
# ------------------------------------------------------------------------------------------------
def find_reference():
    for cand in (os.environ.get("STC_REF_DIR"), "/root/reference/framework", os.path.join(ROOT, "baseline", "_ref", "framework")):
        if cand and os.path.isfile(os.path.join(cand, "STC_GNN.py")):
            return cand
    return None


class ReferenceStack:
    """encoder(2 x T) + decoder(horizon x 2) of the reference with the supports handed in (= STCGNN.forward minus MGP_Gen
    and out_proj, STC_GNN.py:188-204): the same unit of work as stc_gnn_b200.RecurrentStack, same seeded weights."""

    def __init__(self, device, seed=0):
        self.ref_dir = find_reference()
        self.device = device
        torch.manual_seed(seed)
        if self.ref_dir is not None:
            sys.dont_write_bytecode = True
            if self.ref_dir not in sys.path:
                sys.path.insert(0, self.ref_dir)
            import STC_GNN as ref
            self.kind = "reference"
            self.enc = ref.STC_Encoder(SF["N"], SF["C"], SF["Ks"], SF["Kc"], SF["Din"], SF["h"], SF["layers"]).to(device)
            self.dec = ref.STC_Decoder(SF["N"], SF["C"], SF["Ks"], SF["Kc"], SF["h"], SF["h"], SF["layers"], SF["horizon"]).to(device)
            self.leaves = list(self.enc.parameters()) + list(self.dec.parameters())
        else:
            from oracle import stc_oracle as O
            self.kind, self.O = "port", O
            g = torch.Generator().manual_seed(seed)
            self.enc = [O.xavier_cell_params(SF["Din"] if i == 0 else SF["h"], SF["h"], SF["Ks"], SF["Kc"], g, torch.float32)
                        for i in range(SF["layers"])]
            self.dec = [O.xavier_cell_params(SF["h"], SF["h"], SF["Ks"], SF["Kc"], g, torch.float32) for _ in range(SF["layers"])]
            self.leaves = []
            for p in self.enc + self.dec:
                for name in ("Wg", "bg", "Wc", "bc"):
                    t = getattr(p, name).to(device).requires_grad_(True)
                    setattr(p, name, t)
                    self.leaves.append(t)

    def describe(self):
        return ("the unmodified reference's STC_Encoder + STC_Decoder (" + self.ref_dir + ")") if self.kind == "reference" \
            else "oracle/stc_oracle.py reference-shaped port (same operator sequence as BDG_Dif/STC_Cell, autograd)"

    def forward(self, Gs, Gc, X):
        if self.kind == "port":
            return self.O.stack_forward(Gs, Gc, X, self.enc, self.dec, SF["horizon"], SF["Ks"], SF["Kc"],
                                        cell_fn=self.O.stc_cell_refshape)
        _, Ht = self.enc(Gs=Gs, Gc=Gc, X_seq=X, H0_l=None)
        inp, outs = Ht[-1], []
        for _ in range(SF["horizon"]):
            inp, Ht = self.dec(Gs=Gs, Gc=Gc, Xt=inp, H0_l=Ht)
            outs.append(inp)
        return torch.stack(outs, dim=1)

    def step(self, Gs, Gc, X, y):
        for t in self.leaves + [Gs, Gc]:
            t.grad = None
        loss = loss_fn(self.forward(Gs, Gc, X), y)
        loss.backward()
        return loss


def cpu_reference_throughput(B, steps, warmup, seed=0, budget_s=20.0, flush_denormal=False):
    """fwd+bwd samples/s of the reference's cell stack on this box's host cores (fp32, all host threads, autograd) on B
    windows of the same SF-shape workload.  Returns (samples/s, ms/step, timed steps, threads, kind, description)."""
    torch.set_num_threads(os.cpu_count() or 1)
    prev_ftz = torch.set_flush_denormal(bool(flush_denormal))
    try:
        X, y, Gs, Gc = synthetic_inputs(B, seed)
        stack = ReferenceStack("cpu", seed)
        Gs, Gc = Gs.requires_grad_(True), Gc.requires_grad_(True)
        times = []
        t_begin = time.perf_counter()
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            float(stack.step(Gs, Gc, X, y).detach())
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
            if time.perf_counter() - t_begin > budget_s and len(times) >= 2:
                break
    finally:
        torch.set_flush_denormal(False)
    ms = 1e3 * sum(times) / len(times)
    return B / (ms / 1e3), ms, len(times), torch.get_num_threads(), stack.kind, stack.describe()


def cpu_baseline_record(B, steps, warmup, budget_s):
    """The cpu_baseline object: default denormal handling (the reference as shipped) plus the flush-to-zero pair."""
    v, ms, n, cores, kind, what = cpu_reference_throughput(B, steps, warmup, budget_s=budget_s)
    v_ftz, ms_ftz, n_ftz, _, _, _ = cpu_reference_throughput(B, max(2, steps // 2), 1, budget_s=budget_s / 2, flush_denormal=True)
    return {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "ms_per_step": ms, "timed_steps": n,
            "flush_denormal": {"value": v_ftz, "ms_per_step": ms_ftz, "timed_steps": n_ftz},
            "sample": f"{n} timed fwd+bwd steps, each a bounded sample of B={B} windows of the same SF-shape workload "
                      f"(throughput is per window; the benchmark's synthetic supports are denormal-free, so default and "
                      f"torch.set_flush_denormal(True) time the same arithmetic -- the CPU-favourable case); {what}; fp32"}


def run_reference(args, rank):
    if rank != 0:
        return
    rec = cpu_baseline_record(args.cpu_batch, max(2, args.steps), max(0, args.warmup), budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": rec["timed_steps"],
        "warmup": max(0, args.warmup), "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.batch, args.gpus),
        "cpu_baseline": rec,
        "e2e": {"value": rec["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def gpu_eager_baseline(dev, batches, our_step_factory, steps=3):
    """Stock PyTorch eager on this GPU (cuBLAS via einsum, STC_GNN.py:37-42): the reference's cell stack, same seeded
    weights and inputs, fwd+bwd, device-resident, next to this repo's stack at the same batch sizes."""
    rows = []
    stack = ReferenceStack(dev, 0)
    for B in batches:
        row = {"batch": B}
        try:
            X, y, Gs, Gc = synthetic_inputs(B, seed=0)
            X, y = X.to(dev), y.to(dev)
            Gs, Gc = Gs.to(dev).requires_grad_(True), Gc.to(dev).requires_grad_(True)

            def timed(fn, n):
                fn()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(n):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / n

            try:
                ms = timed(lambda: stack.step(Gs, Gc, X, y), steps)
                row.update(eager_samples_per_s=B / (ms / 1e3), eager_ms_per_step=ms,
                           eager_peak_mem_gb=torch.cuda.max_memory_allocated(dev) / 2**30)
            except torch.OutOfMemoryError:
                row["eager_samples_per_s"] = None
                row["eager_note"] = "stock eager ran out of device memory at this batch"
            for t in stack.leaves + [Gs, Gc]:
                t.grad = None
            torch.cuda.empty_cache()
            ours = our_step_factory(B)
            ms_o = timed(ours, max(steps, 5))
            row.update(b200_samples_per_s=B / (ms_o / 1e3), b200_ms_per_step=ms_o)
            if row.get("eager_samples_per_s"):
                row["speedup"] = row["b200_samples_per_s"] / row["eager_samples_per_s"]
        except Exception as exc:   # the baseline sweep must never take the headline down with it
            row["error"] = f"{type(exc).__name__}: {exc}"[:300]
        torch.cuda.empty_cache()
        rows.append(row)
    return {"kind": stack.kind, "what": stack.describe(), "dtype": "f32 (torch default: TF32 off for matmul)",
            "steps_per_point": steps, "sweep": rows}


def workload_config(B, n_gpus, graph=False):
    name = ("sf_cell_stack: encoder 2x9 + decoder 3x2 = 24 STC cell steps/sample, fwd+bwd incl. dGs,dGc "
            "(BASELINE.json configs[1], SF shape)") if WL is SF else (
            "g4096_encoder: 2 layers x T=12 = 24 STC cell steps/sample, fwd+bwd, constant CSR 64x64-grid support and "
            "constant Gc (BASELINE.json configs[2]: N=4096, C=16, F=64)")
    return {
        "workload": name,
        "N": WL["N"], "C": WL["C"], "hidden": WL["h"], "Ks": WL["Ks"], "Kc": WL["Kc"], "layers": WL["layers"],
        "T": WL["T"], "horizon": WL["horizon"], "batch_per_gpu": B, "global_batch": B * n_gpus,
        "parallelism": f"dp{n_gpus}",
        "launch": "cuda-graph replay of the captured step" if graph else "eager (one C-ABI call per cell and direction)",
        "l2": "inputs+activations exceed L2 (no flush needed)" if (B >= 1024 or WL is not SF) else "working set may fit L2",
        "bytes_model": "per-kernel compulsory bytes of the multi-kernel pipeline (DESIGN.md section 4); the fused-cell floor "
                       "of SURVEY 8d is " + ("9.94 MB" if WL is SF else "5.6 GB") + " per sample fwd+bwd",
    }


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def check_dp_parity(stack, leaves, Gs, Gc, bucket, rank, world, dev, b_small=4):
    """Every rank steps on its own shard of a small global batch and all-reduces the flat bucket; every rank also
    steps on the whole concatenated batch alone.  The two gradient sets must agree within the parity tolerance
    (rtol 1e-4 + 5e-5 x mean|ref|: the stack-level floor of tests/test_cell_gpu.py; summation order differs)."""
    import torch.distributed as dist
    shards = [synthetic_inputs(b_small, seed=1000 + r) for r in range(world)]
    Xg = torch.cat([sh[0] for sh in shards]).to(dev)
    yg = torch.cat([sh[1] for sh in shards]).to(dev)

    def grads_of(X, y, scale):
        for p in leaves:
            p.grad = None
        (loss_fn(stack(Gs, Gc, X), y) * scale).backward()

    grads_of(Xg, yg, 1.0)                                   # single process, concatenated batch (mean over world*b)
    want = [p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p) for p in leaves]   # unused cells: no grad
    s, e = rank * b_small, (rank + 1) * b_small
    grads_of(Xg[s:e], yg[s:e], 1.0 / world)                 # shard loss is a mean over b: scale so that the sum is the global mean
    bucket.allreduce()
    ok = True
    for p, w in zip(leaves, want):
        got = p.grad if p.grad is not None else torch.zeros_like(p)
        err = (got.double() - w.double()).abs()
        tol = 1e-4 * w.double().abs() + 5e-5 * w.double().abs().mean()
        ok = ok and bool((err <= tol).all())
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    for p in leaves:
        p.grad = None
    if float(flag.item()) != 1.0:
        raise SystemExit("dp_parity FAILED: bucket-reduced DP gradients differ from the single-process gradients")
    return True


def run_b200(args):
    import torch.distributed as dist
    import stc_gnn_b200 as S
    from stc_gnn_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a GPU (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    _lib.load()

    B = args.batch
    torch.manual_seed(0)
    stack = S.RecurrentStack(WL["N"], WL["C"], WL["Ks"], WL["Kc"], WL["Din"], WL["h"], WL["layers"], WL["horizon"]).to(dev)
    params = list(stack.parameters())
    Xh, yh, Gs_h, Gc_h = synthetic_inputs(B, seed=rank, pin=True)
    if WL is SF:
        Gs = Gs_h.to(dev).requires_grad_(True)
        Gc = Gc_h.to(dev).requires_grad_(True)
        leaves = params + [Gs, Gc]
    else:   # constant supports (no dGs / dGc): 8-neighbour grid scaled by 1/8 as CSR
        from stc_gnn_b200.synth import grid_csr
        rp, ci, va = grid_csr(*WL["grid"])
        Gs = S.CsrSupport(rp.to(dev), ci.to(dev), va.to(dev), WL["N"])
        Gc = Gc_h.to(dev)
        leaves = params
    X_res, y_res = Xh.to(dev), yh.to(dev)
    # data-parallel: one flat fp32 bucket (cell parameters + dGs + dGc), one NCCL all-reduce per step (dp.py)
    bucket = S.dp.GradBucket(leaves) if world > 1 else None

    def allreduce_grads():
        if bucket is not None:
            bucket.allreduce()

    last = {}   # --dump-outputs: the latest step's output and loss (under --cuda-graph, the graph's static tensors)

    def step_loss(X, y):
        out = stack(Gs, Gc, X)
        loss = loss_fn(out, y)
        if args.dump_outputs:   # detached: a kept autograd graph would keep the leaves' AccumulateGrad nodes alive
            last.update(out=out.detach(), loss=loss.detach())
        return loss

    def step(X, y):
        for p in leaves:
            p.grad = None
        loss = step_loss(X, y)
        loss.backward()
        allreduce_grads()
        return loss

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, n):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        sync_all()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- N > 1: bucket-reduced DP gradients == single-process gradients of the concatenated batch (small case,
    #      both through the CUDA path), checked before anything is timed ----
    dp_parity = None
    if world > 1:
        dp_parity = check_dp_parity(stack, leaves, Gs, Gc, bucket, rank, world, dev)

    # ---- device-resident throughput ----
    graphed = None
    if args.cuda_graph:
        if world > 1:
            raise SystemExit("--cuda-graph is a single-GPU option")
        l0 = _lib.LAUNCHES
        step(X_res, y_res)
        per_step_launches = _lib.LAUNCHES - l0
        graphed = S.GraphedStep(step_loss, [X_res, y_res], leaves, warmup=max(args.warmup, 3))
        run_resident = lambda: graphed.replay(X_res, y_res)
    else:
        run_resident = lambda: step(X_res, y_res)
    for _ in range(max(args.warmup, 3)):
        run_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = _lib.LAUNCHES
    ms_total = timed(run_resident, args.steps)
    launches = (per_step_launches * args.steps) if graphed else (_lib.LAUNCHES - l0)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        grads = {f"grad.{n}": p.grad for n, p in stack.named_parameters() if p.grad is not None}   # unused cells: none
        if WL is SF:
            grads.update({"grad.Gs": Gs.grad, "grad.Gc": Gc.grad})
        dump_outputs(args.dump_outputs, {"loss": last["loss"], "out": last["out"], **grads})
    ms_step = ms_total / args.steps
    value = B * world / (ms_step / 1e3)

    # ---- end to end through the module API: pinned host inputs in, loss out, every step ----
    # Every timed step copies one batch of inputs from pinned host memory and reads its loss back.  The copy of step
    # i + 1 is issued on a copy stream right after step i's kernels have been queued (a data loader's prefetch), so it
    # travels under them; the loss read-back still synchronises every step.
    copy_stream = torch.cuda.Stream(device=dev)

    def prefetch():
        with torch.cuda.stream(copy_stream):
            X = Xh.to(dev, non_blocking=True)
            y = yh.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return X, y, ev

    pending = {"next": None}

    def e2e_step():
        if graphed:
            return float(graphed.replay(Xh, yh).item())   # pinned host -> the graph's static inputs, replay, loss out
        if pending["next"] is None:
            pending["next"] = prefetch()
        X, y, ev = pending["next"]
        cur = torch.cuda.current_stream()
        cur.wait_event(ev)
        X.record_stream(cur)
        y.record_stream(cur)
        loss = step(X, y)
        pending["next"] = prefetch()                      # exactly one H2D batch per timed step
        return float(loss.item())

    e2e_step()
    ms_e2e = timed(e2e_step, args.steps) / args.steps
    e2e = {"value": B * world / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": Xh.numel() * 4 + yh.numel() * 4, "d2h_bytes_per_step": 4,
           "note": "inputs copied from pinned host memory every step (next step's copy overlaps this step's kernels), loss read back every step"}
    pending["next"] = None

    # ---- instrumented pass: per-kernel device time + algorithmic bytes over the same K steps ----
    # (every rank runs the pass -- step() contains the gradient all-reduce -- but only rank 0 records and reports)
    roofline, breakdown = None, None
    if rank == 0 and not args.no_roofline:
        _lib.timing_enable(True)
        _lib.timing_collect()
    if not args.no_roofline:
        for _ in range(args.steps):
            step(X_res, y_res)
    sync_all()
    if rank == 0 and not args.no_roofline:
        _lib.timing_enable(False)
        kinds = _lib.timing_collect()
        peak, peak_src = measured_peaks()
        tot_ms = sum(v[0] for v in kinds.values())
        breakdown = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps,
                         "share": v[0] / tot_ms, "achieved_GBs": v[2] / (v[0] * 1e-3) / 1e9}
                     for k, v in sorted(kinds.items(), key=lambda kv: -kv[1][0])}
        top = max(kinds.items(), key=lambda kv: kv[1][0])
        name, (kms, kn, kbytes) = top
        achieved = kbytes / (kms * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic(name) if (WL is SF and B == 4096) else (None, None)
        roofline = {"kernel": name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                    "avg_launch_us": 1e3 * kms / kn, "alg_bytes_per_launch": kbytes / kn,
                    "share_of_kernel_time": kms / tot_ms,
                    "note": "achieved = this kernel's own compulsory bytes (inputs it must read + outputs it must write, "
                            "formula beside its launcher) / its mean launch time over every launch of the step (both "
                            "convolutions, Din = 1 and Din = 16 cells); 3xTF32 tcgen05 kernel (see DESIGN.md section 4)"}

    # ---- the whole step against the fused-cell floor of SURVEY 8d (ALG_BYTES_TRAIN = 4 N C (3 Din + 11 h) per
    #      cell-step-sample: what a fully fused cell must move, forward incl. saving u,r,c + backward) ----
    roofline_step = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        n_enc0 = WL["T"]                                              # layer-0 encoder cells: Din = input width
        n_wide = WL["T"] * (WL["layers"] - 1) + WL["horizon"] * WL["layers"]
        per_sample = 4.0 * WL["N"] * WL["C"] * (n_enc0 * (3 * WL["Din"] + 11 * WL["h"]) + n_wide * (3 * WL["h"] + 11 * WL["h"]))
        ach = per_sample * B / (ms_step * 1e-3) / 1e9
        roofline_step = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "alg_bytes_per_sample": per_sample, "peak_source": peak_src,
                         "bytes_model": "SURVEY 8d ALG_BYTES_TRAIN summed over the cell steps of one sample "
                                        "(compulsory traffic of a fully fused cell), x batch / device step time (per GPU)"}

    cpu_baseline, eager = None, None
    if rank == 0 and world == 1 and WL is SF:
        if not args.no_eager_baseline:
            def ours_at(Bq):
                Xq, yq, _, _ = synthetic_inputs(Bq, seed=0)
                Xq, yq = Xq.to(dev), yq.to(dev)
                return lambda: step(Xq, yq)
            eager = gpu_eager_baseline(dev, [32, 512, 4096], ours_at)
            # the reference's own batch size replayed from a CUDA graph (an eager step of 48 C-ABI calls is host-bound there)
            try:
                Xq, yq, _, _ = synthetic_inputs(32, seed=0)
                Xq, yq = Xq.to(dev), yq.to(dev)
                gs32 = S.GraphedStep(lambda X, y: loss_fn(stack(Gs, Gc, X), y), [Xq, yq], leaves, warmup=3)
                for _ in range(3):
                    gs32.replay(Xq, yq)
                torch.cuda.synchronize()
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                for _ in range(20):
                    gs32.replay(Xq, yq)
                g1.record()
                torch.cuda.synchronize()
                ms32 = g0.elapsed_time(g1) / 20
                eager["graph_replay_b32"] = {"batch": 32, "b200_samples_per_s": 32 / (ms32 / 1e3), "b200_ms_per_step": ms32,
                                             "what": "stc_gnn_b200.GraphedStep replay of the same fwd+bwd step"}
                del gs32
            except Exception as exc:
                eager["graph_replay_b32"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
            for p in leaves:
                p.grad = None
        if not args.no_cpu_baseline:
            cpu_baseline = cpu_baseline_record(args.cpu_batch, 40, 1, budget_s=14.0)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(B, world, graph=bool(graphed)),
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_step": roofline_step,
            "cpu_baseline": cpu_baseline, "gpu_eager_baseline": eager, "dp_parity": dp_parity,
            "kernel_breakdown": breakdown,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    global WL, METRIC
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    if args.workload == "g4096":
        WL = G4096
        METRIC = "train samples/s (fwd+bwd), N=4096 C=16 F=64 STC encoder stack"
        if args.batch == 4096:
            args.batch = 4
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "no CPU arm for the g4096 side workload"}), flush=True)
            return
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_b200(args)


if __name__ == "__main__":
    main()
