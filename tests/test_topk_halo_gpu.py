"""The sparse generator choosing its pattern on the row-partitioned graph, on the GPU: the row-block selection
(stc_pair_topk_rows, `pair_topk(..., rows=)`) bitwise against the full selection and against fp64, its workspace, timing
kind and C-ABI error paths; `PartitionedSupport.k_regular` on the device (the host constructor's fields, one
synchronising copy); `SparseGraphGenerator(...)(X_seq, k=k, partition=RowPartition(...))` at world 1 (bitwise the
unpartitioned selection partitioned afterwards; a partitioned RecurrentStack fed with it bitwise in its output) and at
world 2 and 3 over gloo with every rank on one GPU, and over NCCL when two GPUs are visible.

Selection margin and tolerances are those of tests/test_topk_graph_gpu.py and tests/test_halo_sparse_mgp_gpu.py: the
references of P and the gradients are the fp32 unpartitioned generator on the selected pattern on the same GPU."""
import os
import socket
import traceback
import warnings

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from stc_gnn_b200 import _lib, dp, halo
from stc_gnn_b200.halo import PartitionedSupport, RowPartition
from tests import sparse_mgp_oracle as SO
from tests import topk_graph_oracle as TO
from tests.test_sparse_mgp_gpu import GEN_FLOOR, STACK_FLOOR
from tests.test_topk_halo_cpu import assert_same_partition, host_partition, random_selection

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def uv(N, W, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.tanh(torch.randn(N, W, generator=g)).to(DEV), torch.tanh(torch.randn(N, W, generator=g)).to(DEV))


def blocks(N):
    """Row blocks (row0, n_rows): row0 not a multiple of 128, one row, the last partial block, a block over several
    128-row blocks."""
    cand = [(N - 1, 1), (0, 1), (3, N - 3), (N // 3, N // 3 + 1), (N - min(N, 130), min(N, 130)), (5, min(N - 5, 700))]
    return [(r, n) for r, n in cand if r >= 0 and n >= 1 and r + n <= N]


# ---- 1. the row-block kernel ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W", [4, 36, 384])
@pytest.mark.parametrize("N", [7, 129, 300, 1000, 4096])
def test_row_blocks_are_rows_of_the_full_selection(N, W):
    U, V = uv(N, W, 7 * N + W)
    S64 = TO.full_scores(U.double(), V.double())
    for k in (1, 8, 32):
        if k > N:
            continue
        cols, sc = S.pair_topk(U, V, k, scores=True)
        for r0, n in blocks(N):
            tag = f"(N {N}, W {W}, k {k}, rows [{r0}, {r0} + {n}))"
            c, s = S.pair_topk(U, V, k, scores=True, rows=(r0, n))
            assert c.shape == (n, k) and s.shape == (n, k), tag
            assert torch.equal(c, cols[r0:r0 + n]) and torch.equal(s, sc[r0:r0 + n]), f"not bitwise the full rows {tag}"
            assert torch.equal(S.pair_topk(U, V, k, rows=(r0, n)), c), f"without scores {tag}"
            c2, s2 = S.pair_topk(U, V, k, scores=True, rows=(r0, n))
            assert torch.equal(c, c2) and torch.equal(s, s2), f"two calls differ {tag}"
            TO.check_selection(S64[r0:r0 + n], c, k)
    empty = S.pair_topk(U, V, 1, rows=(N // 2, 0))
    assert empty.shape == (0, 1)


def test_config4_row_block_against_fp64_and_peak_memory():
    """N = 65,536, width 384, a rank's n_rows = 8,192 (world 8) starting at a row that is not a multiple of 128: 256
    sampled rows against fp64 scores over all columns, bitwise the full selection's rows, and the peak memory of a call
    is the workspace plus the outputs."""
    N, W, k, n = 65536, 384, 16, 8192
    r0 = 5 * n + 77
    U, V = uv(N, W, 8)
    lib = _lib.load()
    ws = lib.stc_pair_topk_rows_workspace_bytes(N, W, n, k)
    nseg = ws // (8 * n * k)
    assert ws == nseg * n * k * 8 and nseg > 1, (ws, nseg)   # 64 row blocks: the columns split into segments
    assert ws < lib.stc_pair_topk_workspace_bytes(N, W, k)
    cols, sc = S.pair_topk(U, V, k, scores=True, rows=(r0, n))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    cols2, sc2 = S.pair_topk(U, V, k, scores=True, rows=(r0, n))
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak <= ws + 8 * n * k + (1 << 20), (peak, ws)
    assert torch.equal(cols, cols2) and torch.equal(sc, sc2)
    del cols2, sc2
    full, fsc = S.pair_topk(U, V, k, scores=True)
    assert torch.equal(full[r0:r0 + n], cols) and torch.equal(fsc[r0:r0 + n], sc)
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(1))[:256].to(DEV)
    S64 = TO.full_scores(U.double(), V.double(), rows + r0)
    near = TO.check_selection(S64, cols[rows], k)
    O.assert_close(sc[rows].double().cpu(), S64.gather(1, cols[rows].long()).cpu(), "scores (config 4 row block)")
    print(f"config 4 row block: {nseg} segments, {near} near-tie rows of 256")


def test_row_block_timing_kind():
    U, V = uv(512, 64, 3)
    _lib.timing_enable(True)
    _lib.timing_collect()
    S.pair_topk(U, V, 8, rows=(100, 300))
    S.pair_topk(U, V, 8)
    torch.cuda.synchronize()
    _lib.timing_enable(False)
    kinds = _lib.timing_collect()
    assert kinds["pair_topk_rows"][1] == 1 and kinds["pair_topk_rows"][2] == 8.0 * 512 * 64 + 8.0 * 300 * 8, kinds
    assert kinds["pair_topk"][1] == 1, kinds


def test_row_block_error_paths_return_before_a_launch():
    lib = _lib.load()
    N, W = 20, 8
    U = torch.zeros(N, W, device=DEV)
    cols = torch.empty(N, 32, dtype=torch.int32, device=DEV)
    ws = torch.empty(1 << 20, dtype=torch.uint8, device=DEV)
    st = torch.cuda.current_stream().cuda_stream

    def call(k=4, row0=2, n=10, width=W, nbytes=1 << 20, u=U.data_ptr(), c=cols.data_ptr(), w=ws.data_ptr()):
        status = lib.stc_pair_topk_rows(N, width, u, U.data_ptr(), row0, n, k, c, None, w, nbytes, st)
        return status, lib.stc_last_launch_count()

    assert call(k=33) == (-2, 0) and b"at most 32" in lib.stc_last_error()
    for bad in (dict(k=0), dict(k=21), dict(width=6), dict(row0=-1), dict(n=-1), dict(row0=15, n=6), dict(u=None),
                dict(c=None), dict(w=None), dict(u=U.data_ptr() + 4), dict(w=ws.data_ptr() + 4)):
        assert call(**bad) == (-1, 0), bad
    assert call(nbytes=16) == (-3, 0)
    assert call(n=0, u=None, c=None, w=None) == (0, 0), "n_rows = 0 launches nothing"
    assert call() == (0, 2)
    assert lib.stc_pair_topk_rows_workspace_bytes(N, W, 0, 4) == 0
    assert lib.stc_pair_topk_rows_workspace_bytes(N, W, N + 1, 4) == 0
    assert lib.stc_pair_topk_rows_workspace_bytes(N, W, 5, 33) == 0
    assert lib.stc_pair_topk_rows_workspace_bytes(N, W, N, 4) == lib.stc_pair_topk_workspace_bytes(N, W, 4)
    with pytest.raises(RuntimeError, match="outside"):
        S.pair_topk(U, U, 4, rows=(15, 6))
    with pytest.raises(RuntimeError, match="outside"):
        S.pair_topk(U, U, 4, rows=(-1, 3))


# ---- 2. the partition of a selection, built on the device ------------------------------------------------------------
def _to_cpu(ps):
    """The device-built partition's tensors on the host, for comparison with the host constructor."""
    cp = lambda t: t.cpu()
    out = PartitionedSupport.__new__(PartitionedSupport)
    out.__dict__.update(ps.__dict__)
    out._rowptr, out._col = cp(ps._rowptr), cp(ps._col)
    for d in ("fwd", "bwd"):
        p = getattr(ps, d)
        setattr(out, d, halo.HaloPlan(rank=p.rank, world=p.world, start=p.start, nloc=p.nloc, nhalo=p.nhalo,
                                      send_idx=[cp(t) for t in p.send_idx], recv_counts=p.recv_counts,
                                      halo_global=cp(p.halo_global), op_row=cp(p.op_row), op_col=cp(p.op_col),
                                      op_val=cp(p.op_val)))
    m = ps.maps()
    maps = halo.ValueMaps(**{f: (cp(v) if isinstance(v, torch.Tensor) else v) for f, v in m.__dict__.items()})
    out._dev = {"maps": maps}
    for d in ("fwd", "bwd"):
        st = ps._device_state(d, DEV)
        out._dev[("xchg", d, "cpu")] = {"send_idx": cp(st["send_idx"]), "nsend": st["nsend"],
                                       "interior": cp(st["interior"]), "boundary": cp(st["boundary"]), "buffers": {}}
    return out


@pytest.mark.parametrize("N,k", [(61, 4), (300, 8), (7, 1)])
def test_device_builder_is_the_host_partition(N, k):
    for world in (1, 2, 3, 4):
        cols = random_selection(N, k, N + world)
        for rank in range(world):
            got = PartitionedSupport.k_regular(cols.to(DEV), rank, world)
            assert got.maps().fwd_ids.is_cuda and got.fwd.send_idx[0].is_cuda
            assert_same_partition(_to_cpu(got), host_partition(cols, rank, world), f"(N {N}, k {k}, {rank}/{world})")


def test_device_builder_synchronises_once():
    N, k, world = 4096, 16, 4
    U, V = uv(N, 64, 2)
    cols = S.pair_topk(U, V, k)
    part = RowPartition(N, 1, world)
    part.support(cols)                              # warm-up: kernels loaded, allocator primed
    torch.cuda.synchronize()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            ps = part.support(cols)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    syncs = [w for w in caught if "called a synchronizing" in str(w.message)]
    assert len(syncs) == 1, [str(w.message) for w in syncs]
    assert ps.fwd.nhalo > 0 and len(part._streams) == 0, "building creates no stream"


# ---- 3. world 1 ---------------------------------------------------------------------------------------------------------
def _problem(N, B, T, C, hg, seed):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(B, T, N, C, generator=g)
    torch.manual_seed(seed)
    return X, S.SparseGraphGenerator(C, hg)


@pytest.mark.parametrize("N,k", [(90, 8), (300, 16)])
def test_world_one_is_the_selection_partitioned_afterwards(N, k):
    B, T, C, hg = 2, 3, 3, 4
    X, gen = _problem(N, B, T, C, hg, seed=N + k)
    gen = gen.to(DEV)
    w = torch.randn(N * k, generator=torch.Generator().manual_seed(k)).to(DEV)
    res = []
    for mode in ("after", "partition"):
        gen.zero_grad(set_to_none=True)
        Xd = X.to(DEV).requires_grad_(True)
        if mode == "after":
            cs = gen(Xd, k=k)
            sup = PartitionedSupport.from_csr_support(cs, 0, 1)
            assert sup.vals is cs.vals
        else:
            sup = gen(Xd, k=k, partition=RowPartition(N, 0, 1))
        assert isinstance(sup, PartitionedSupport) and sup.learnable
        (sup.vals * w).sum().backward()
        torch.cuda.synchronize()
        res.append([sup._col.to(DEV).long(), sup.vals.detach(), gen.params_S["Wu"].grad, gen.params_S["Wv"].grad,
                    Xd.grad])
    for name, a, b in zip(("columns", "P", "dWu", "dWv", "dX_seq"), *res):
        assert torch.equal(a, b), f"{name} differs (N {N}, k {k})"


@pytest.mark.parametrize("Ks", [2, 4])
def test_world_one_stack(Ks):
    """The stack's output is bitwise; its gradients are compared with the stack floor, because the adjoint hops add the
    edge gradient with atomics (one per batch sample and column chunk of an edge), so the gradient arriving at P, and
    everything computed from it, is not bitwise repeatable even between two runs of the same path."""
    N, C, Kc, h, layers, horizon, B, T, hg, k = 64, 3, 2, 8, 2, 2, 2, 3, 4, 8
    X, gen = _problem(N, B, T, C, hg, seed=60 + Ks)
    gen = gen.to(DEV)
    torch.manual_seed(Ks)
    stack = S.RecurrentStack(N, C, Ks, Kc, 1, h, layers, horizon).to(DEV)
    g = torch.Generator().manual_seed(Ks)
    Gc = (torch.rand(C, C, generator=g) / C).to(DEV)
    dOut = torch.randn(B, horizon, N, C, h, generator=g).to(DEV)
    res = []
    for mode in ("after", "partition"):
        gen.zero_grad(set_to_none=True)
        stack.zero_grad(set_to_none=True)
        Xd = X.to(DEV).requires_grad_(True)
        sup = (PartitionedSupport.from_csr_support(gen(Xd, k=k), 0, 1) if mode == "after"
               else gen(Xd, k=k, partition=RowPartition(N, 0, 1)))
        out = stack(sup, Gc, Xd[..., None])
        out.backward(dOut)
        torch.cuda.synchronize()
        res.append([out.detach(), Xd.grad] + [p.grad for p in list(gen.parameters()) + list(stack.parameters())])
    assert torch.equal(res[0][0], res[1][0]), f"stack output (Ks {Ks})"
    for i, (a, b) in enumerate(zip(*res)):
        O.assert_close(a.cpu(), b.cpu(), f"stack tensor {i} (Ks {Ks})", atol_scale=STACK_FLOOR)


def test_no_grad_partition_support_is_constant():
    N, k = 50, 4
    X, gen = _problem(N, 2, 3, 3, 4, seed=5)
    gen = gen.to(DEV)
    with torch.no_grad():
        sup = gen(X.to(DEV), k=k, partition=RowPartition(N, 0, 1))
    assert not sup.vals.requires_grad
    assert torch.equal(sup.vals, gen(X.to(DEV), k=k).vals.detach())


def test_partition_error_paths():
    N = 20
    gen = S.SparseGraphGenerator(4, 8).to(DEV)
    X = torch.randn(2, 3, N, 4, device=DEV)
    part = RowPartition(N, 0, 1)
    ps = PartitionedSupport.k_regular(random_selection(N, 4, 0).to(DEV), 0, 1)
    with pytest.raises(RuntimeError, match="give k="):
        gen(X, partition=part)
    with pytest.raises(RuntimeError, match="give k="):
        gen(X, ps, k=4, partition=part)
    with pytest.raises(RuntimeError, match="row partition"):
        gen(X, k=4, partition=part, group=object())
    with pytest.raises(RuntimeError, match="row partition"):
        gen(X, k=4, partition=part, average=True)
    with pytest.raises(RuntimeError, match="halo.RowPartition"):
        gen(X, k=4, partition=ps)
    with pytest.raises(RuntimeError, match="has 20 nodes, the input 21"):
        gen(torch.randn(2, 3, 21, 4, device=DEV), k=4, partition=part)
    with pytest.raises(RuntimeError, match="outside"):
        gen(X, k=21, partition=part)
    # unchanged: a fixed partitioned pattern and k stay exclusive, k= and batch data-parallelism too
    with pytest.raises(RuntimeError, match="row-partitioned"):
        gen(X, ps, k=4)
    with pytest.raises(RuntimeError, match="batch data-parallelism"):
        gen(X, k=4, group=object())


# ---- 4. several ranks ----------------------------------------------------------------------------------------------------
def _generator_case(rank, world, dev):
    """The selection (same bytes on every rank, bitwise pair_topk of the gathered U, V, fp64 margin), P, dWu / dWv
    (reduce_per_cell True, and False with a GradBucket) and this rank's dX_seq against the unpartitioned generator on
    the selected pattern, and the error paths before any collective."""
    single = [dist.new_group([r]) for r in range(world)][rank]     # the references run without collectives
    for N, k in ((61, 8), (47, 4)):
        B, T, C, hg = 2, 3, 3, 4
        X, gen = _problem(N, B, T, C, hg, seed=N)
        gen = gen.to(dev)
        w = torch.randn(N * k, generator=torch.Generator().manual_seed(N)).to(dev)
        part = RowPartition(N, rank, world)
        lo, n = part.start, part.nloc
        Xd = X.to(dev)
        for per_cell in (True, False):
            part.reduce_per_cell = per_cell
            gen.zero_grad(set_to_none=True)
            Xl = Xd[:, :, lo:lo + n].contiguous().requires_grad_(True)
            sup = gen(Xl, k=k, partition=part)
            assert isinstance(sup, PartitionedSupport) and sup.reduce_per_cell == per_cell
            (sup.vals * w).sum().backward()
            if not per_cell:
                dp.GradBucket(list(gen.parameters())).allreduce()
            torch.cuda.synchronize()
            got = {"P": sup.vals.detach(), "dWu": gen.params_S["Wu"].grad.clone(),
                   "dWv": gen.params_S["Wv"].grad.clone(), "dX": Xl.grad}
            tag = f"(N {N}, k {k}, rank {rank}/{world}, reduce_per_cell {per_cell})"
            cols = sup._col.view(N, k).to(torch.int32)
            other = cols.clone()
            dist.broadcast(other, 0)
            assert torch.equal(other, cols), f"the selection is the same bytes on every rank {tag}"
            # this rank's rows: bitwise pair_topk of the gathered U, V
            with torch.no_grad():
                Xn = Xl.detach().permute(2, 0, 1, 3).reshape(n, B * T, C)
                U = torch.tanh(gen.alpha * (Xn @ gen.params_S["Wu"])).reshape(n, -1)
                V = torch.tanh(gen.alpha * (Xn @ gen.params_S["Wv"])).reshape(n, -1)
                UV = part.gather_rows(torch.cat([U, V], 1))
                W = U.shape[1]
                assert torch.equal(S.pair_topk(UV[:, :W], UV[:, W:], k), cols), f"not pair_topk of the gathered U, V {tag}"
                U64 = SO.node_major(X.double(), gen.params_S["Wu"].detach().double().cpu(), gen.alpha)
                V64 = SO.node_major(X.double(), gen.params_S["Wv"].detach().double().cpu(), gen.alpha)
                TO.check_selection(TO.full_scores(U64, V64), cols.cpu(), k)
            # the unpartitioned generator on the selected pattern
            gen.zero_grad(set_to_none=True)
            Xr = Xd.clone().requires_grad_(True)
            fixed = S.CsrSupport((torch.arange(N + 1, device=dev) * k).int(), cols.reshape(-1),
                                 torch.ones(N * k, device=dev), N)
            ref = gen(Xr, fixed, group=single)
            (ref.vals * w).sum().backward()
            torch.cuda.synchronize()
            O.assert_close(got["P"].cpu(), ref.vals.detach().cpu(), f"P {tag}")
            for name in ("Wu", "Wv"):
                O.assert_close(got["d" + name].cpu(), gen.params_S[name].grad.cpu(), f"d{name} {tag}",
                               atol_scale=GEN_FLOOR)
            O.assert_close(got["dX"].cpu(), Xr.grad[:, :, lo:lo + n].cpu(), f"dX_seq {tag}")
    # the new error paths raise on every rank before any collective
    gen = S.SparseGraphGenerator(3, 4).to(dev)
    part = RowPartition(61, rank, world)
    Xl = torch.randn(2, 3, part.nloc, 3, device=dev)
    for kw in (dict(), dict(k=4, group=single), dict(k=4, average=True)):
        with pytest.raises(RuntimeError):
            gen(Xl, partition=part, **kw)
    dist.barrier()


def _stack_case(rank, world, dev):
    """A selected partitioned support feeding a partitioned RecurrentStack (Ks 2 and 3) == the unpartitioned generator
    on the selected pattern + stack: outputs, dWu, dWv, the stack's parameters (one GradBucket per step) and dX_seq."""
    N, C, Kc, h, layers, horizon, B, T, hg, k = 47, 3, 2, 8, 2, 2, 2, 3, 4, 6
    single = [dist.new_group([r]) for r in range(world)][rank]
    for Ks in (2, 3):
        X, gen = _problem(N, B, T, C, hg, seed=70 + Ks)
        gen = gen.to(dev)
        torch.manual_seed(70 + Ks)
        stack = S.RecurrentStack(N, C, Ks, Kc, 1, h, layers, horizon).to(dev)
        g = torch.Generator().manual_seed(80 + Ks)
        Gc = (torch.rand(C, C, generator=g) / C).to(dev)
        dOut = torch.randn(B, horizon, N, C, h, generator=g).to(dev)
        part = RowPartition(N, rank, world)
        part.reduce_per_cell = False
        lo, n = part.start, part.nloc
        loc = S.RecurrentStack(n, C, Ks, Kc, 1, h, layers, horizon).to(dev)
        loc.load_state_dict(stack.state_dict())
        Xl = X.to(dev)[:, :, lo:lo + n].contiguous().requires_grad_(True)
        sup = gen(Xl, k=k, partition=part)
        out_l = loc(sup, Gc, Xl[..., None])
        out_l.backward(dOut[:, :, lo:lo + n])
        lparams = list(gen.parameters()) + list(loc.parameters())
        dp.GradBucket(lparams).allreduce()
        torch.cuda.synchronize()
        got = [out_l.detach(), Xl.grad] + [p.grad.clone() for p in lparams]
        gen.zero_grad(set_to_none=True)
        fixed = S.CsrSupport((torch.arange(N + 1, device=dev) * k).int(), sup._col.to(torch.int32),
                             torch.ones(N * k, device=dev), N)
        Xd = X.to(dev).requires_grad_(True)
        out = stack(gen(Xd, fixed, group=single), Gc, Xd[..., None])
        out.backward(dOut)
        torch.cuda.synchronize()
        want = [out.detach()[:, :, lo:lo + n], Xd.grad[:, :, lo:lo + n]] + \
            [p.grad for p in list(gen.parameters()) + list(stack.parameters())]
        for i, (a, b) in enumerate(zip(got, want)):
            O.assert_close(a.cpu(), b.cpu(), f"stack tensor {i} (rank {rank}/{world}, Ks {Ks})", atol_scale=STACK_FLOOR)


def _worker(rank, world, port, backend, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        dev = torch.device("cuda", rank if backend == "nccl" else 0)
        torch.cuda.set_device(dev)
        if backend == "nccl":
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        else:
            dist.init_process_group("gloo", rank=rank, world_size=world)
        _generator_case(rank, world, dev)
        _stack_case(rank, world, dev)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, None))
    except Exception:  # pragma: no cover - reported by the parent
        q.put((rank, traceback.format_exc()))


def _run_ranks(backend, world):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, backend, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        results = [q.get(timeout=300) for _ in procs]
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
                p.join(timeout=10)
    errs = [f"rank {r}:\n{e}" for r, e in results if e]
    assert not errs, "\n".join(errs)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_selected_partition_two_ranks_nccl():
    _run_ranks("nccl", 2)


def test_selected_partition_two_ranks_gloo_one_gpu():
    _run_ranks("gloo", 2)


def test_selected_partition_three_ranks_gloo_one_gpu():
    _run_ranks("gloo", 3)
