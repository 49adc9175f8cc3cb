"""The graph generator on a row-partitioned pattern, on the GPU: the row-list scores kernel
(stc_pair_scores_csr_rows), `SparseGraphGenerator` on a `halo.PartitionedSupport` against the unpartitioned generator
(bitwise at world 1; at world 2 and 3 over gloo with every rank on one GPU, and over NCCL when two GPUs are visible),
a generated partitioned support feeding a partitioned RecurrentStack, the no-grad path, the scores launches of a
rank, and the error paths.

Tolerances and floors are those of tests/test_sparse_mgp_gpu.py: |got - ref| <= 1e-4 * |ref| + 1e-5 * mean|ref|, and
GEN_FLOOR = 5e-5 * mean|ref| for the Wu / Wv gradients (STACK_FLOOR through a stack).  The references here are the
fp32 unpartitioned generator and stack on the same GPU."""
import os
import socket
import traceback

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from stc_gnn_b200 import _lib, dp
from stc_gnn_b200.halo import PartitionedSupport
from tests import sparse_mgp_oracle as SO
from tests.test_sparse_mgp_gpu import GEN_FLOOR, STACK_FLOOR, csr, safe

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _scores_rows(pat, width, ld, U, V, Sc, rows):
    st = torch.cuda.current_stream().cuda_stream
    return _lib.load().stc_pair_scores_csr_rows(pat.struct(), pat.N, width, ld, U.data_ptr(), V.data_ptr(),
                                                Sc.data_ptr(), rows.data_ptr() if rows is not None else None,
                                                0 if rows is None else rows.numel(), st)


# ---- 1. the row-list kernel ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("width", [1, 3, 4, 384, 1100])
def test_row_list_scores_kernel(width):
    N = 300
    g = torch.Generator().manual_seed(width)
    rowptr, col = SO.random_pattern(N, 9, seed=width, empty_every=7, hub=(40, 120))
    pat = csr(rowptr, col)
    ld = 2 * width + 4                                  # U and V side by side in one buffer, rows padded
    UV = torch.randn(N, ld, generator=g).to(DEV)
    U, V = UV[:, :width], UV[:, width:2 * width]
    plain = torch.empty(pat.nnz, device=DEV)
    Uc, Vc = U.contiguous(), V.contiguous()             # the plain kernel's separate [N, width] operands
    _lib.check(_lib.load().stc_pair_scores_csr(pat.struct(), N, width, Uc.data_ptr(), Vc.data_ptr(), plain.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream), "stc_pair_scores_csr")
    listed = torch.zeros(N, dtype=torch.bool)
    listed[torch.randperm(N, generator=g)[:N // 3]] = True
    listed[40] = listed[1] = True                       # the hub row and an empty row
    rows = torch.nonzero(listed).flatten().to(torch.int32).to(DEV)
    buf = torch.full((pat.nnz + 64,), 7.0, device=DEV)  # canary in every unlisted entry and past nnz
    Sc = buf[:pat.nnz]
    assert _scores_rows(pat, width, ld, U, V, Sc, rows) == 0
    assert _lib.last_launch_count() == 1
    torch.cuda.synchronize()
    mine = listed[SO.edge_rows(rowptr)].to(DEV)
    assert torch.equal(Sc[mine], plain[mine]), "listed rows: bitwise the plain kernel"
    assert bool((Sc[~mine] == 7.0).all()) and bool((buf[pat.nnz:] == 7.0).all()), "nothing else is written"
    rest = torch.nonzero(~listed).flatten().to(torch.int32).to(DEV)
    assert _scores_rows(pat, width, ld, U, V, Sc, rest) == 0
    torch.cuda.synchronize()
    assert torch.equal(Sc, plain), "interior list + boundary list == the plain kernel"
    # an empty list launches nothing
    before = buf.clone()
    assert _lib.load().stc_pair_scores_csr_rows(pat.struct(), N, width, ld, U.data_ptr(), V.data_ptr(), Sc.data_ptr(),
                                                rows.data_ptr(), 0, torch.cuda.current_stream().cuda_stream) == 0
    assert _lib.last_launch_count() == 0
    torch.cuda.synchronize()
    assert torch.equal(buf, before)
    # error codes
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    call = lambda gs=pat.struct(), n=N, w=width, l=ld, r=rows.data_ptr(), k=rows.numel(): \
        lib.stc_pair_scores_csr_rows(gs, n, w, l, U.data_ptr(), V.data_ptr(), Sc.data_ptr(), r, k, st)
    assert call(l=width - 1) == -1 and b"ld" in lib.stc_last_error()
    assert call(w=0, l=4) == -1
    assert call(r=None) == -1
    assert call(k=N + 1) == -1 and call(k=-1) == -1
    assert call(n=0) == -1
    assert call(gs=S.support.dense_struct(torch.zeros(N, N, device=DEV))) == -2 and b"CSR" in lib.stc_last_error()


# ---- helpers -------------------------------------------------------------------------------------------------------
def _problem(N, B, T, C, hg, seed, deg=6, empty_every=7):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(B, T, N, C, generator=g)
    torch.manual_seed(seed)
    gen = S.SparseGraphGenerator(C, hg)
    rowptr, col = SO.random_pattern(N, deg, seed=seed, empty_every=empty_every)
    with torch.no_grad():
        rowptr, col = safe(rowptr, col, SO.node_major(X.double(), gen.params_S["Wu"].double(), gen.alpha),
                           SO.node_major(X.double(), gen.params_S["Wv"].double(), gen.alpha))
    w = torch.randn(col.numel(), generator=g)
    return X, gen, rowptr, col, w


def _partition(rowptr, col, N, rank, world):
    vals = torch.rand(col.numel(), generator=torch.Generator().manual_seed(0))
    return PartitionedSupport(rowptr.long(), col.long(), vals, N, rank, world)


# ---- 2. world 1: bitwise the unpartitioned generator ---------------------------------------------------------------
@pytest.mark.parametrize("B,T,hg", [(2, 3, 4), (1, 1, 3)])
def test_world_one_is_bitwise_the_unpartitioned_generator(B, T, hg):
    N, C = 90, 3
    X, gen, rowptr, col, w = _problem(N, B, T, C, hg, seed=11 + hg)
    gen = gen.to(DEV)
    res = []
    for pattern in (csr(rowptr, col), _partition(rowptr, col, N, 0, 1)):
        gen.zero_grad(set_to_none=True)
        Xd = X.to(DEV).requires_grad_(True)
        sup = gen(Xd, pattern)
        assert type(sup) is type(pattern) and sup.learnable
        (sup.vals * w.to(DEV)).sum().backward()
        torch.cuda.synchronize()
        res.append([sup.vals.detach(), gen.params_S["Wu"].grad, gen.params_S["Wv"].grad, Xd.grad])
    for name, a, b in zip(("P", "dWu", "dWv", "dX_seq"), *res):
        assert torch.equal(a, b), f"{name} differs from the unpartitioned generator (B {B}, T {T}, hg {hg})"


# ---- 5. no-grad: a constant support for the cell -------------------------------------------------------------------
def test_no_grad_partitioned_support_launches_no_gradient_hop():
    N, B, T, C, hg, h, Ks, Kc = 64, 2, 3, 3, 4, 8, 3, 2
    X, gen, rowptr, col, _ = _problem(N, B, T, C, hg, seed=6)
    gen = gen.to(DEV)
    ps = _partition(rowptr, col, N, 0, 1)
    with torch.no_grad():
        sup = gen(X.to(DEV), ps)
    assert not sup.vals.requires_grad
    assert torch.equal(sup.vals, gen(X.to(DEV), csr(rowptr, col)).vals.detach())
    cell = S.STC_Cell(N, C, Ks, Kc, 1, h).to(DEV)
    g = torch.Generator().manual_seed(6)
    Gc = (torch.rand(C, C, generator=g) / C).to(DEV)
    Xt = torch.randn(B, N, C, 1, generator=g).to(DEV)
    H = torch.randn(B, N, C, h, generator=g).to(DEV).requires_grad_(True)
    _lib.timing_enable(True)
    _lib.timing_collect()
    cell(Gs=sup, Gc=Gc, Xt=Xt, Ht_1=H).sum().backward()
    torch.cuda.synchronize()
    _lib.timing_enable(False)
    kinds = _lib.timing_collect()
    assert "support_csr_grad" not in kinds and kinds["support_csr"][1] > 0, kinds
    assert gen.params_S["Wu"].grad is None and H.grad is not None


# ---- 7. error paths --------------------------------------------------------------------------------------------------
def test_error_paths_on_a_partitioned_pattern():
    N = 20
    gen = S.SparseGraphGenerator(4, 8).to(DEV)
    rowptr, col = SO.random_pattern(N, 4, seed=1)
    ps = _partition(rowptr, col, N, 0, 1)
    X = torch.randn(2, 3, N, 4, device=DEV)
    with pytest.raises(RuntimeError, match="cannot be combined"):
        gen(X, ps, group=object())
    with pytest.raises(RuntimeError, match="cannot be combined"):
        gen(X, ps, average=True)
    with pytest.raises(RuntimeError, match="block of the pattern has 20 nodes, the input 21"):
        gen(torch.randn(2, 3, 21, 4, device=DEV), ps)
    with pytest.raises(RuntimeError, match="CsrSupport"):
        gen(X, torch.zeros(N, N, device=DEV))
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.pair_softmax_partitioned(torch.zeros(N, 6), torch.zeros(N, 6), ps)


# ---- 3, 4, 6. several ranks ------------------------------------------------------------------------------------------
def _generator_case(rank, world, dev):
    """P on every rank, the Wu / Wv gradients (reduce_per_cell True, and False with a GradBucket) and this rank's
    block of dX_seq against the unpartitioned generator; N = 61 is not a multiple of 2 or 3, rows are empty."""
    N, B, T, C, hg = 61, 2, 3, 3, 4
    single = [dist.new_group([r]) for r in range(world)][rank]     # the reference runs without collectives
    X, gen, rowptr, col, w = _problem(N, B, T, C, hg, seed=21)
    gen = gen.to(dev)
    Xd = X.to(dev).requires_grad_(True)
    ref = gen(Xd, csr(rowptr, col, dev), group=single)
    (ref.vals * w.to(dev)).sum().backward()
    want = {"P": ref.vals.detach(), "dWu": gen.params_S["Wu"].grad.clone(), "dWv": gen.params_S["Wv"].grad.clone()}
    ps = _partition(rowptr, col, N, rank, world)
    assert ps.fwd.nhalo > 0
    lo, n = ps.start, ps.nloc
    for per_cell in (True, False):
        ps.reduce_per_cell = per_cell
        gen.zero_grad(set_to_none=True)
        Xl = Xd.detach()[:, :, lo:lo + n].contiguous().requires_grad_(True)
        sup = gen(Xl, ps)
        assert isinstance(sup, PartitionedSupport) and sup.vals.shape == (ps.nnz,)
        (sup.vals * w.to(dev)).sum().backward()
        if not per_cell:
            dp.GradBucket(list(gen.parameters())).allreduce()
        torch.cuda.synchronize()
        tag = f"(rank {rank}/{world}, reduce_per_cell {per_cell})"
        O.assert_close(sup.vals.detach().cpu(), want["P"].cpu(), f"P {tag}")
        other = sup.vals.detach().clone()
        dist.broadcast(other, 0)
        assert torch.equal(other, sup.vals.detach()), "P is the same bytes on every rank"
        for k in ("Wu", "Wv"):
            O.assert_close(gen.params_S[k].grad.cpu(), want["d" + k].cpu(), f"d{k} {tag}", atol_scale=GEN_FLOOR)
        O.assert_close(Xl.grad.cpu(), Xd.grad[:, :, lo:lo + n].cpu(), f"dX_seq {tag}")
    # 6. a rank's scores launches cover its own rows only (interior + boundary)
    ps.reduce_per_cell = True
    Xl = Xd.detach()[:, :, lo:lo + n].contiguous()
    kinds = {}
    for name, pattern, x in (("part", ps, Xl), ("full", csr(rowptr, col, dev), Xd.detach())):
        _lib.timing_enable(True)
        _lib.timing_collect()
        with torch.no_grad():
            gen(x, pattern, group=single if name == "full" else None)
        torch.cuda.synchronize()
        _lib.timing_enable(False)
        kinds[name] = _lib.timing_collect()["pair_scores_csr"]
    assert kinds["full"][1] == 1 and 1 <= kinds["part"][1] <= 2, kinds
    assert kinds["part"][2] < 0.8 * kinds["full"][2], kinds


def _stack_case(rank, world, dev):
    """A generated partitioned support feeding a partitioned RecurrentStack (Ks 2 and 3) == the unpartitioned
    generator + stack: outputs, dWu, dWv, the stack's parameters (one GradBucket per step) and dX_seq."""
    N, C, Kc, h, layers, horizon, B, T, hg = 47, 3, 2, 8, 2, 2, 2, 3, 4
    single = [dist.new_group([r]) for r in range(world)][rank] if world > 1 else None
    for Ks in (2, 3):
        X, gen, rowptr, col, _ = _problem(N, B, T, C, hg, seed=40 + Ks)
        gen = gen.to(dev)
        torch.manual_seed(40 + Ks)
        stack = S.RecurrentStack(N, C, Ks, Kc, 1, h, layers, horizon).to(dev)
        g = torch.Generator().manual_seed(50 + Ks)
        Gc = (torch.rand(C, C, generator=g) / C).to(dev)
        dOut = torch.randn(B, horizon, N, C, h, generator=g).to(dev)
        Xd = X.to(dev).requires_grad_(True)
        out = stack(gen(Xd, csr(rowptr, col, dev), group=single), Gc, Xd[..., None])
        out.backward(dOut)
        params = list(gen.parameters()) + list(stack.parameters())
        want = [out.detach(), Xd.grad.clone()] + [p.grad.clone() for p in params]
        ps = _partition(rowptr, col, N, rank, world)
        ps.reduce_per_cell = False
        lo, n = ps.start, ps.nloc
        loc = S.RecurrentStack(n, C, Ks, Kc, 1, h, layers, horizon).to(dev)
        loc.load_state_dict(stack.state_dict())
        gen.zero_grad(set_to_none=True)
        Xl = Xd.detach()[:, :, lo:lo + n].contiguous().requires_grad_(True)
        out_l = loc(gen(Xl, ps), Gc, Xl[..., None])
        out_l.backward(dOut[:, :, lo:lo + n])
        lparams = list(gen.parameters()) + list(loc.parameters())
        dp.GradBucket(lparams).allreduce()
        torch.cuda.synchronize()
        got = [out_l.detach(), Xl.grad] + [p.grad for p in lparams]
        want[0], want[1] = want[0][:, :, lo:lo + n], want[1][:, :, lo:lo + n]
        for i, (a, b) in enumerate(zip(got, want)):
            O.assert_close(a.cpu(), b.cpu(), f"stack tensor {i} (rank {rank}/{world}, Ks {Ks})",
                           atol_scale=STACK_FLOOR)


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


def test_generated_stack_world_one():
    _stack_case(0, 1, torch.device(DEV))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_partitioned_generator_two_ranks_nccl():
    _run_ranks("nccl", 2)


def test_partitioned_generator_two_ranks_gloo_one_gpu():
    _run_ranks("gloo", 2)


def test_partitioned_generator_three_ranks_gloo_one_gpu():
    _run_ranks("gloo", 3)
