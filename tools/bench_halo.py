#!/usr/bin/env python
"""BASELINE configs[3]: one STC cell forward on the N = 65,536 kNN graph (C = 8, F = 64, Ks = 4 = 3 hops), nodes
row-partitioned over the ranks with a halo exchange per hop (stc_gnn_b200/halo.py).  Launch under torchrun:

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/bench_halo.py [B] [--train]

`--train`: forward + backward of the cell (gradients w.r.t. Xt, H, Gc and the parameters; the partitioned backward runs
the adjoint hops with their own halo exchanges; the parameter gradients are all-reduced ONCE per step in a flat bucket,
`--reduce-per-cell` restores one all-reduce per cell backward).  At world > 1 every rank first checks its block of the
partitioned result (outputs and every gradient) against the unpartitioned cell run on the same GPU -> `parity_ok`.

Strong scaling: the global problem is fixed, each rank owns N / world nodes.  Time = max over ranks (CUDA events,
barrier on both sides).  Rank 0 prints one JSON line.

`--train --learned`: the same training step with learnable edge values (an `nn.Parameter` [nnz] behind the
partitioned support, its gradient formed inside the adjoint hops) and with the constant support, in one process,
alternating ROUNDS times; both reduce their gradients once per step in a flat bucket (the learnable one also holds
the [nnz] edge gradient).  It runs the partitioned path at every world size, world 1 included, and reports
median / min / max ms of each, their ratio, nnz, the bucket sizes, and the device's name, power limit and maximum SM
clock.  At world > 1, `parity_ok` also covers the edge gradient against the unpartitioned learnable cell.
`--train --generated`: the config 4 step with the spatial support generated from the input window on the kNN pattern
(`SparseGraphGenerator` on the partitioned pattern, X_seq [B, T = 12, N, C], hg = 16) in front of the partitioned cell,
against the learnable partitioned step on fixed values, alternating as `--learned` does; also the generator's own
forward + backward per rank.  At world > 1, `parity_ok` covers P, the Wu / Wv / X_seq gradients and the cell outputs
against the unpartitioned generator + cell on the same GPU, and over NCCL the replicated form (X_seq all-gathered, the
whole generator on every rank, its [nnz] gradient all-reduced) is timed as well.
`--gloo`: every rank on cuda:0, exchanging over gloo -- a full-size parity check of the partitioned path on a
machine with one GPU; its times measure ranks sharing one GPU, not scaling."""
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import stc_gnn_b200 as S  # noqa: E402
from stc_gnn_b200 import _lib  # noqa: E402
from stc_gnn_b200.halo import PartitionedSupport, partitioned_cell_forward  # noqa: E402
from stc_gnn_b200.synth import knn_csr  # noqa: E402


def violations(got, ref, atol_scale):
    got, ref = got.double(), ref.double()
    scale = ref.abs().mean()
    err = (got - ref).abs()
    return int((err > 1e-4 * ref.abs() + atol_scale * scale).sum()), float(err.max() / scale)


def learned_main(B, world, rank, dev):
    """--train --learned: learnable vs constant partitioned training step (see the module docstring)."""
    N, C, F, Ks, Kc, ROUNDS, iters = 65536, 8, 64, 4, 2, 7, 10
    rp, ci, va = knn_csr(N, 8)
    torch.manual_seed(0)
    cell = S.STC_Cell(N, C, Ks, Kc, F, F).to(dev)
    params = list(cell.parameters())
    Gc = (torch.rand(C, C, generator=torch.Generator().manual_seed(1)) / C).to(dev).requires_grad_(True)
    g = torch.Generator().manual_seed(100)
    Xg = torch.randn(B, N, C, F, generator=g)
    Hg = torch.randn(B, N, C, F, generator=g) * 0.5
    dHg = torch.randn(B, N, C, F, generator=g)
    # non-uniform values, identical on every rank (one seed)
    vals = torch.nn.Parameter((va * (0.5 + torch.rand(va.numel(), generator=torch.Generator().manual_seed(7)))).to(dev))
    const = PartitionedSupport(rp, ci, vals.detach().cpu(), N, rank, world)
    learned = const.with_values(vals)
    lo, n = const.start, const.nloc
    blk = lambda t: t[:, lo:lo + n].contiguous().to(dev)
    X, H, dHn = blk(Xg).requires_grad_(True), blk(Hg).requires_grad_(True), blk(dHg)
    buckets = {"constant": S.dp.GradBucket(params + [Gc]), "learnable": S.dp.GradBucket(params + [Gc, vals])}
    sups = {"constant": const, "learnable": learned}

    def step(which):
        def run():
            for t in (X, H, vals, Gc, *params):
                t.grad = None
            out = partitioned_cell_forward(sups[which], Gc, X, H, cell.gates.W, cell.gates.b, cell.candi.W,
                                           cell.candi.b, Ks, Kc, reduce_params=False)
            out.backward(dHn)
            buckets[which].allreduce()       # ONE gradient all-reduce per step (a no-op at world 1)
            return out
        return run

    variants = {k: step(k) for k in sups}
    parity = None
    if world > 1:
        # this rank's block of the partitioned result == the unpartitioned learnable cell on the same GPU
        out_p = variants["learnable"]().detach().clone()
        got = [out_p, X.grad.clone(), H.grad.clone()] + [t.grad.clone() for t in params + [Gc, vals]]
        full = S.CsrSupport(rp.to(dev), ci.to(dev), vals, N)
        Xf, Hf = Xg.to(dev).requires_grad_(True), Hg.to(dev).requires_grad_(True)
        for t in params + [Gc, vals]:
            t.grad = None
        out_f = cell(Gs=full, Gc=Gc, Xt=Xf, Ht_1=Hf)
        out_f.backward(dHg.to(dev))
        want = [out_f.detach()[:, lo:lo + n], Xf.grad[:, lo:lo + n], Hf.grad[:, lo:lo + n]] + \
               [t.grad.clone() for t in params + [Gc, vals]]
        names = ["H'", "dXt", "dH", "dWg", "dbg", "dWc", "dbc", "dGc", "dvals"]
        worst, nbad = {}, 0
        for nm, a_, b_ in zip(names, got, want):
            # reduced gradients sum B*N*C = 1 M rows (dvals: B*C*F = 1,024 products per edge) in another order
            nb, w = violations(a_, b_, 1e-5 if nm in ("H'", "dXt", "dH") else 3e-5)
            worst[nm] = w
            nbad += nb
        flag = torch.tensor([float(nbad)], device=dev)
        dist.all_reduce(flag)
        parity = {"parity_ok": float(flag.item()) == 0.0, "worst_err_over_mean_ref_rank0": worst}
        del Xf, Hf, out_f, want, got, full
        torch.cuda.empty_cache()

    for fn in variants.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    samples = {k: [] for k in variants}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(ROUNDS):
        for k, fn in variants.items():
            if world > 1:
                dist.barrier()
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            samples[k].append(e0.elapsed_time(e1) / iters)
    if world > 1:                            # time of a round = the slowest rank's
        for k in samples:
            t = torch.tensor(samples[k], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            samples[k] = t.tolist()
    if rank == 0:
        try:
            smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        except Exception as e:  # the measurement still stands, but says that the limit is unknown
            smi = f"unavailable: {e!r}"
        summ = lambda v: {"median": statistics.median(v), "min": min(v), "max": max(v)}
        backend = dist.get_backend() if world > 1 else None
        rec = {"kind": "config4_cell_step_partitioned_learned", "n_gpus": 1 if backend in (None, "gloo") else world,
               "n_ranks": world, "backend": backend, "device": torch.cuda.get_device_name(dev),
               "power_limit_and_max_sm_clock": smi, "N": N, "C": C, "F": F, "Ks": Ks, "Kc": Kc, "B": B, "nnz": learned.nnz,
               "local_rows": n, "fwd_halo_rows": const.fwd.nhalo, "rounds": ROUNDS, "steps_per_round": iters,
               "constant_ms": summ(samples["constant"]), "learnable_ms": summ(samples["learnable"]),
               "ratio_learnable_over_constant": statistics.median(samples["learnable"]) / statistics.median(samples["constant"]),
               "bucket_floats_constant": buckets["constant"].numel, "bucket_floats_learnable": buckets["learnable"].numel}
        if parity:
            rec.update(parity)
        print(json.dumps(rec), flush=True)


def _device_record(dev):
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the measurement still stands, but says that the limit is unknown
        smi = f"unavailable: {e!r}"
    return {"device": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": smi}


def _alternate(variants, world, rounds, iters):
    """{name: [ms per step of each round]}, the variants alternating, a round's time the slowest rank's."""
    for fn in variants.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    samples = {k: [] for k in variants}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for k, fn in variants.items():
            if world > 1:
                dist.barrier()
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            samples[k].append(e0.elapsed_time(e1) / iters)
    if world > 1:
        for k in samples:
            t = torch.tensor(samples[k], device=torch.cuda.current_device())
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            samples[k] = t.tolist()
    return samples


def generated_main(B, world, rank, dev):
    """--train --generated: generator + partitioned step vs the learnable partitioned step (see the module docstring)."""
    N, C, F, Ks, Kc, T, hg, ROUNDS, iters = 65536, 8, 64, 4, 2, 12, 16, 7, 10
    rp, ci, va = knn_csr(N, 8)
    torch.manual_seed(0)
    cell = S.STC_Cell(N, C, Ks, Kc, F, F).to(dev)
    gen = S.SparseGraphGenerator(C, hg).to(dev)
    params, gparams = list(cell.parameters()), list(gen.parameters())
    Gc = (torch.rand(C, C, generator=torch.Generator().manual_seed(1)) / C).to(dev).requires_grad_(True)
    g = torch.Generator().manual_seed(100)
    Xg = torch.randn(B, N, C, F, generator=g)
    Hg = torch.randn(B, N, C, F, generator=g) * 0.5
    dHg = torch.randn(B, N, C, F, generator=g)
    Xsg = torch.randn(B, T, N, C, generator=g)
    vals = torch.nn.Parameter((va * (0.5 + torch.rand(va.numel(), generator=torch.Generator().manual_seed(7)))).to(dev))
    const = PartitionedSupport(rp, ci, vals.detach().cpu(), N, rank, world)
    const.reduce_per_cell = False            # every gradient goes through one bucket per step
    learned = const.with_values(vals)
    lo, n = const.start, const.nloc
    blk = lambda t, d=1: t.narrow(d, lo, n).contiguous().to(dev)
    X, H, dHn = blk(Xg).requires_grad_(True), blk(Hg).requires_grad_(True), blk(dHg)
    Xs = blk(Xsg, 2).requires_grad_(True)
    wP = torch.randn(learned.nnz, generator=torch.Generator().manual_seed(5)).to(dev)
    buckets = {"learnable": S.dp.GradBucket(params + [Gc, vals]), "generated": S.dp.GradBucket(params + [Gc] + gparams)}
    cell_args = lambda: (Gc, X, H, cell.gates.W, cell.gates.b, cell.candi.W, cell.candi.b, Ks, Kc)
    # one-rank groups: the unpartitioned generator runs without batch-DP collectives
    singles = [dist.new_group([r]) for r in range(world)] if world > 1 else [None]

    def clear():
        for t in (X, H, Xs, vals, Gc, *params, *gparams):
            t.grad = None

    def learnable_step():
        clear()
        out = partitioned_cell_forward(learned, *cell_args(), reduce_params=False)
        out.backward(dHn)
        buckets["learnable"].allreduce()
        return out

    def generated_step():
        clear()
        sup = gen(Xs, const)
        out = partitioned_cell_forward(sup, *cell_args(), reduce_params=False)
        out.backward(dHn)
        buckets["generated"].allreduce()
        return out, sup

    def generator_only():
        clear()
        (gen(Xs, const).vals * wP).sum().backward()

    variants = {"learnable": learnable_step, "generated": lambda: generated_step()[0]}
    if world > 1 and dist.get_backend() == "nccl":
        # the replicated form: every rank gathers the whole window and runs the whole generator; the [nnz] gradient
        # arriving at P must then be all-reduced (mgp.reduce_grad) before the generator's backward
        cs = S.CsrSupport(rp.to(dev), ci.to(dev), va.to(dev), N)
        rep_bucket = S.dp.GradBucket(params + [Gc])

        def replicated_step():
            clear()
            parts = [torch.empty_like(Xs) for _ in range(world)]
            dist.all_gather(parts, Xs.detach())
            Xfull = torch.cat(parts, dim=2)
            P = S.mgp.reduce_grad(gen(Xfull, cs, group=singles[rank]).vals)
            out = partitioned_cell_forward(const.with_values(P), *cell_args(), reduce_params=False)
            out.backward(dHn)
            rep_bucket.allreduce()
            return out
        variants["replicated"] = replicated_step

    parity = None
    if world > 1:
        out_p, sup = generated_step()
        got = [sup.vals.detach().clone(), out_p.detach().clone(), X.grad.clone(), H.grad.clone(), Xs.grad.clone()] + \
              [t.grad.clone() for t in gparams + params + [Gc]]
        clear()
        full = S.CsrSupport(rp.to(dev), ci.to(dev), va.to(dev), N)
        Xf, Hf, Xsf = (t.to(dev).requires_grad_(True) for t in (Xg, Hg, Xsg))
        gsup = gen(Xsf, full, group=singles[rank])
        out_f = cell(Gs=gsup, Gc=Gc, Xt=Xf, Ht_1=Hf)
        out_f.backward(dHg.to(dev))
        want = [gsup.vals.detach(), out_f.detach()[:, lo:lo + n], Xf.grad[:, lo:lo + n], Hf.grad[:, lo:lo + n],
                Xsf.grad[:, :, lo:lo + n]] + [t.grad.clone() for t in gparams + params + [Gc]]
        names = ["P", "H'", "dXt", "dH", "dX_seq", "dWu", "dWv", "dWg", "dbg", "dWc", "dbc", "dGc"]
        floors = {"P": 1e-5, "H'": 1e-5, "dXt": 1e-5, "dH": 1e-5, "dX_seq": 1e-5, "dWu": 5e-5, "dWv": 5e-5}
        worst, nbad = {}, 0
        m = const.maps()
        for nm, a_, b_ in zip(names, got, want):
            if nm == "P":            # this rank's rows, and the whole vector every rank holds
                nb, worst["P_own_rows"] = violations(a_[m.edge_lo:m.edge_hi], b_[m.edge_lo:m.edge_hi], 1e-5)
                nbad += nb
            nb, worst[nm] = violations(a_, b_, floors.get(nm, 3e-5))
            nbad += nb
        flag = torch.tensor([float(nbad)], device=dev)
        dist.all_reduce(flag)
        parity = {"parity_ok": float(flag.item()) == 0.0, "worst_err_over_mean_ref_rank0": worst}
        del Xf, Hf, Xsf, gsup, out_f, want, got, full, sup, out_p
        clear()
        torch.cuda.empty_cache()

    gen_only = _alternate({"generator": generator_only}, world, 3, iters)["generator"]
    samples = _alternate(variants, world, ROUNDS, iters)
    if rank == 0:
        summ = lambda v: {"median": statistics.median(v), "min": min(v), "max": max(v)}
        backend = dist.get_backend() if world > 1 else None
        rec = {"kind": "config4_cell_step_partitioned_generated", "n_gpus": 1 if backend in (None, "gloo") else world,
               "n_ranks": world, "backend": backend, **_device_record(dev), "N": N, "C": C, "F": F, "Ks": Ks,
               "Kc": Kc, "B": B, "T": T, "hg": hg, "nnz": learned.nnz, "local_rows": n,
               "fwd_halo_rows": const.fwd.nhalo, "rounds": ROUNDS, "steps_per_round": iters,
               "generator_fwd_bwd_ms": summ(gen_only)}
        rec.update({f"{k}_step_ms": summ(v) for k, v in samples.items()})
        med = {k: statistics.median(v) for k, v in samples.items()}
        rec["ratio_generated_over_learnable"] = med["generated"] / med["learnable"]
        if "replicated" in med:
            rec["ratio_generated_over_replicated"] = med["generated"] / med["replicated"]
        if parity:
            rec.update(parity)
        print(json.dumps(rec), flush=True)


def main():
    train = "--train" in sys.argv
    per_cell = "--reduce-per-cell" in sys.argv
    pos = [a for a in sys.argv[1:] if not a.startswith("--")]
    B = int(pos[0]) if pos else 2
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    gloo = "--gloo" in sys.argv
    local = 0 if gloo else int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if gloo:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    if "--generated" in sys.argv:
        if not train:
            raise SystemExit("--generated measures the training step: pass --train as well")
        generated_main(B, world, rank, dev)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    if "--learned" in sys.argv:
        if not train:
            raise SystemExit("--learned measures the training step: pass --train as well")
        learned_main(B, world, rank, dev)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    N, C, F, Ks, Kc = 65536, 8, 64, 4, 2
    rp, ci, va = knn_csr(N, 8)
    torch.manual_seed(0)
    cell = S.STC_Cell(N, C, Ks, Kc, F, F).to(dev)
    params = list(cell.parameters())
    Gc = (torch.rand(C, C, generator=torch.Generator().manual_seed(1)) / C).to(dev)
    # the GLOBAL problem is generated identically on every rank (one seed); a rank keeps its node block
    g = torch.Generator().manual_seed(100)
    Xg = torch.randn(B, N, C, F, generator=g)
    Hg = torch.randn(B, N, C, F, generator=g) * 0.5
    dHg = torch.randn(B, N, C, F, generator=g)
    full = S.CsrSupport(rp.to(dev), ci.to(dev), va.to(dev), N)
    with torch.set_grad_enabled(train):
        if world > 1:
            ps = PartitionedSupport(rp, ci, va, N, rank, world)
            ps.reduce_per_cell = per_cell
            lo, n = ps.start, ps.nloc
            halo = {"fwd_halo_rows": ps.fwd.nhalo, "local_rows": n}
        else:
            ps, lo, n = full, 0, N
            halo = {"fwd_halo_rows": 0, "local_rows": n}
        blk = lambda t: t[:, lo:lo + n].contiguous().to(dev)
        X, H, dHn = blk(Xg).requires_grad_(train), blk(Hg).requires_grad_(train), blk(dHg)
        Gc.requires_grad_(train)
        leaves = params + [Gc]
        bucket = S.dp.GradBucket(leaves) if (world > 1 and train and not per_cell) else None

        def fwd():
            if world > 1:
                return partitioned_cell_forward(ps, Gc, X, H, cell.gates.W, cell.gates.b, cell.candi.W, cell.candi.b, Ks, Kc,
                                                reduce_params=per_cell)
            return cell(Gs=ps, Gc=Gc, Xt=X, Ht_1=H)

        def step():
            out = fwd()
            if train:
                for t in (X, H, *leaves):
                    t.grad = None
                out.backward(dHn)
                if bucket is not None:
                    bucket.allreduce()        # ONE parameter-gradient all-reduce per step
            return out

        # ---- parity: this rank's block of the partitioned result == the unpartitioned result on the same GPU ----
        parity = None
        if world > 1:
            out_p = step().detach().clone()
            got = [out_p] + ([X.grad.clone(), H.grad.clone()] + [t.grad.clone() for t in leaves] if train else [])
            Xf, Hf = Xg.to(dev).requires_grad_(train), Hg.to(dev).requires_grad_(train)
            for t in leaves:
                t.grad = None
            out_f = cell(Gs=full, Gc=Gc, Xt=Xf, Ht_1=Hf)
            want = [out_f.detach()[:, lo:lo + n]]
            if train:
                out_f.backward(dHg.to(dev))
                want += [Xf.grad[:, lo:lo + n], Hf.grad[:, lo:lo + n]] + [t.grad.clone() for t in leaves]
            names = ["H'", "dXt", "dH", "dWg", "dbg", "dWc", "dbc", "dGc"]
            worst, nbad = {}, 0
            for nm, a_, b_ in zip(names, got, want):
                # parameter gradients sum B*N*C = 1 M rows in a different order: the dW floor of tests/test_cell_gpu.py
                nb, w = violations(a_, b_, 3e-5 if nm.startswith("dW") or nm.startswith("db") or nm == "dGc" else 1e-5)
                worst[nm] = w
                nbad += nb
            flag = torch.tensor([float(nbad)], device=dev)
            dist.all_reduce(flag)
            parity = {"parity_ok": float(flag.item()) == 0.0, "worst_err_over_mean_ref_rank0": worst}
            del Xf, Hf, out_f, want, got
            torch.cuda.empty_cache()

        for _ in range(3):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 10
        e0.record()
        for _ in range(iters):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
    if rank == 0:
        rec = {"kind": "config4_cell_step_partitioned" if train else "config4_cell_fwd_partitioned", "n_gpus": world, "N": N,
               "C": C, "F": F, "Ks": Ks, "B": B, "ms": ms, "cell_step_samples_per_s": B / ms * 1e3, "scaling": "strong",
               "param_allreduce": ("per cell backward" if per_cell else "once per step (flat bucket)") if train else None,
               "exchange": "side stream: device pack -> NCCL all-to-all -> device unpack, interior rows computed meanwhile",
               **halo}
        if parity:
            rec.update(parity)
        print(json.dumps(rec), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
