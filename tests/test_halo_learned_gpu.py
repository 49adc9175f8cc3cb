"""Learnable edge values on a row-partitioned CSR support, on the GPU: the fused edge-gradient hop over a row list
(stc_support_apply_rows_edge_grad), `PartitionedSupport.hop_ext` against the unpartitioned learnable `CsrSupport`, the
partitioned cell and a stack against the fp64 oracle, in-place and non-leaf values, and two ranks (NCCL over two GPUs,
or gloo with both ranks on one GPU).

Tolerance as everywhere: |got - ref| <= 1e-4 * |ref| + 1e-5 * mean|ref| per cell, 5e-5 * mean|ref| through a stack."""
import os
import socket
import traceback

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from tests.helpers import oracle_cell_with_grads, random_case
from tests.learned_csr_oracle import stc_cell_edge_grad
from tests.test_learned_csr_gpu import dense_of, edge_rows, pattern

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ARGS = ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")


# ---- 1. the fused hop over a row list ----------------------------------------------------------------------------
@pytest.mark.parametrize("width", [1, 5, 64, 512])
@pytest.mark.parametrize("B", [1, 3])
def test_row_list_fused_hop(width, B):
    N = 300
    rowptr, col, vals = pattern(N, 8, seed=width + 10 * B, empty_every=7, hub=(40, 250))
    sup = S.CsrSupport(rowptr.to(DEV), col.to(DEV), vals.to(DEV), N)
    g = torch.Generator().manual_seed(width + B)
    X, Z = (torch.randn(B, N, width, generator=g).to(DEV) for _ in range(2))
    A = torch.randn(B, 2, N, width, generator=g).to(DEV)[:, 1]            # batch-strided, per-sample slab contiguous
    listed = torch.zeros(N, dtype=torch.bool)
    listed[torch.randperm(N, generator=g)[:N // 3]] = True
    listed[40] = listed[1] = True                                          # the hub row and an empty row
    rows = torch.nonzero(listed).flatten().to(torch.int32).to(DEV)
    rest = torch.nonzero(~listed).flatten().to(torch.int32).to(DEV)
    coef = 2.0
    buf = torch.zeros(sup.nnz + 64, device=DEV)
    buf[sup.nnz:] = 12345.0                                                # canary after dvals[nnz]
    dvals = buf[:sup.nnz]
    out = torch.full((B, N, width), 7.0, device=DEV)
    S.support_apply_edge_grad(sup, X, A, dvals, coef=coef, alpha=coef, beta=1.0, Z=Z, out=out, rows=rows)
    plain = torch.full((B, N, width), 7.0, device=DEV)
    S.support_apply(sup, X, transpose=False, alpha=coef, beta=1.0, Z=Z, out=plain, rows=rows)
    torch.cuda.synchronize()
    assert torch.equal(out, plain), "listed rows: what the plain row-list hop writes; other rows untouched"
    assert bool((out[:, ~listed.to(DEV)] == 7.0).all())
    assert bool((buf[sup.nnz:] == 12345.0).all()), "nothing past dvals[nnz] may be written"
    r, c = edge_rows(rowptr), col.long()
    mine = listed[r]
    ref = coef * (A.double().cpu()[:, r] * X.double().cpu()[:, c]).sum(dim=(0, 2)) * mine
    O.assert_close(dvals.cpu(), ref, f"dvals of the listed rows W={width} B={B}")
    assert not dvals.cpu()[~mine].any(), "edges of unlisted rows get no gradient"
    # interior list + boundary list == the full fused hop (in-place accumulation form, out aliases Z)
    acc, d_split = Z.clone(), torch.zeros(sup.nnz, device=DEV)
    for lst in (rows, rest):
        S.support_apply_edge_grad(sup, X, A, d_split, coef=coef, alpha=coef, beta=1.0, Z=acc, out=acc, rows=lst)
    d_full = torch.zeros(sup.nnz, device=DEV)
    full = S.support_apply_edge_grad(sup, X, A, d_full, coef=coef, alpha=coef, beta=1.0, Z=Z)
    torch.cuda.synchronize()
    assert torch.equal(acc, full)
    torch.testing.assert_close(d_split, d_full)
    with pytest.raises(RuntimeError, match="needs `out`"):
        S.support_apply_edge_grad(sup, X, A, d_full, rows=rows)


# ---- helpers -------------------------------------------------------------------------------------------------------
def learnable_partition(rowptr, col, vals, N, rank, world, dev=DEV):
    v = torch.nn.Parameter(vals.float().to(dev))
    return S.halo.PartitionedSupport(rowptr, col, v, N, rank, world), v


def _learned_cell_block(rank, world, dev, shape, seed, check_ranks_agree=False):
    """Partitioned cell with learnable values on this rank's block == the unpartitioned fp64 oracle: H', every
    gradient and the [nnz] edge gradient (all-reduced: the full gradient on every rank)."""
    B, N, C, Din, h, Ks, Kc = shape
    rowptr, col, vals = pattern(N, 6, seed=seed, empty_every=9)
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=seed)
    t["Gs"] = dense_of(rowptr, col, vals, N)
    Hn_o, g_o = oracle_cell_with_grads(t, dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc))
    dv_o = stc_cell_edge_grad(torch.sparse_csr_tensor(rowptr.long(), col.long(), vals.double(), size=(N, N)),
                              *(t[k] for k in ARGS), Ks, Kc, t["dHn"])
    ps, v = learnable_partition(rowptr, col, vals, N, rank, world, dev)
    loc = lambda k: ps.local_slice(t[k]) if k in ("Xt", "H", "dHn") else t[k]
    p = {k: loc(k).float().to(dev).requires_grad_(True) for k in ARGS}
    out = S.halo.partitioned_cell_forward(ps, *(p[k] for k in ARGS), Ks, Kc)
    out.backward(loc("dHn").float().to(dev))
    torch.cuda.synchronize()
    tag = f"(rank {rank}/{world}, Ks {Ks}, Kc {Kc})"
    O.assert_close(out.detach().cpu(), ps.local_slice(Hn_o), f"H' {tag}")
    O.assert_close(v.grad.cpu(), dv_o, f"dvals {tag}")
    for k, name in (("Xt", "dXt"), ("H", "dH")):
        O.assert_close(p[k].grad.cpu(), ps.local_slice(g_o[name]), f"{name} {tag}")
    for k, name in (("Wg", "dWg"), ("Wc", "dWc"), ("bg", "dbg"), ("bc", "dbc"), ("Gc", "dGc")):
        O.assert_close(p[k].grad.cpu(), g_o[name], f"{name} {tag}")
    if check_ranks_agree:
        other = v.grad.clone()
        dist.broadcast(other, 0)
        assert torch.equal(other, v.grad), "every rank holds the same reduced edge gradient"
    return ps


# ---- 2. world-1 partitioned cell -----------------------------------------------------------------------------------
@pytest.mark.parametrize("Ks", [1, 2, 3, 4])
@pytest.mark.parametrize("Kc", [1, 2, 3])
def test_single_rank_learnable_partitioned_cell(Ks, Kc):
    _learned_cell_block(0, 1, torch.device(DEV), (2, 60, 3, 4, 8, Ks, Kc), seed=Ks * 5 + Kc)


# ---- 3. hop_ext == the unpartitioned learnable CsrSupport -----------------------------------------------------------
def test_hop_ext_matches_unpartitioned_learnable_support():
    N, B, W = 200, 2, 24
    rowptr, col, vals = pattern(N, 7, seed=4, empty_every=5, hub=(3, 150))
    v = torch.nn.Parameter(vals.float().to(DEV))
    cs = S.CsrSupport(rowptr.to(DEV), col.to(DEV), v, N)
    ps = S.halo.PartitionedSupport.from_csr_support(cs, 0, 1)
    assert ps.learnable and ps.vals is cs.vals
    g = torch.Generator().manual_seed(5)
    X, Z, A = (torch.randn(B, N, W, generator=g).to(DEV) for _ in range(3))
    ps.sync_values(X.device)
    for direction, tr in (("fwd", True), ("bwd", False)):
        out = torch.empty_like(X)
        ps.hop_ext(X, out, Z_ext=Z, alpha=2.0, beta=-1.0, direction=direction)
        assert torch.equal(out, S.support_apply(cs, X, transpose=tr, alpha=2.0, beta=-1.0, Z=Z)), direction
    d1, d2 = torch.zeros(cs.nnz, device=DEV), torch.zeros(cs.nnz, device=DEV)
    out = Z.clone()
    ps.hop_ext(X, out, Z_ext=out, alpha=2.0, beta=1.0, direction="bwd", A_ext=A, coef=2.0, dvals=d1)
    want = S.support_apply_edge_grad(cs, X, A, d2, coef=2.0, alpha=2.0, beta=1.0, Z=Z)
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    torch.testing.assert_close(d1, d2)
    with pytest.raises(RuntimeError, match="edge gradient needs"):
        ps.hop_ext(X, out, direction="fwd", A_ext=A, dvals=d1)


# ---- 4. a stack: partitioned (per-step reduction through a GradBucket) == unpartitioned ----------------------------
def test_recurrent_stack_on_a_learnable_partitioned_support():
    N, C, Din, h, Ks, Kc, T, B = 40, 3, 2, 8, 3, 2, 3, 2
    rowptr, col, vals = pattern(N, 5, seed=12, empty_every=8)
    torch.manual_seed(3)
    stack = S.RecurrentStack(N, C, Ks, Kc, Din, h, 2, 2).to(DEV)
    g = torch.Generator().manual_seed(8)
    X = torch.randn(B, T, N, C, Din, generator=g).to(DEV)
    dOut = torch.randn(B, 2, N, C, h, generator=g).to(DEV)
    Gc0 = (torch.rand(C, C, generator=g) / C).to(DEV)
    res = []
    for partitioned in (False, True):
        v = torch.nn.Parameter(vals.float().to(DEV))
        cs = S.CsrSupport(rowptr.to(DEV), col.to(DEV), v, N)
        Gs = S.halo.PartitionedSupport.from_csr_support(cs, 0, 1) if partitioned else cs
        if partitioned:
            Gs.reduce_per_cell = False
        Gc = Gc0.clone().requires_grad_(True)
        stack.zero_grad(set_to_none=True)
        out = stack(Gs, Gc, X)
        out.backward(dOut)
        if partitioned:
            S.dp.GradBucket(list(stack.parameters()) + [Gc, v]).allreduce()
        res.append([out.detach(), Gc.grad, v.grad] + [p.grad.clone() for p in stack.parameters()])
    for i, (a, b) in enumerate(zip(*res)):
        O.assert_close(b.cpu(), a.double().cpu(), f"stack tensor {i}: partitioned vs CSR support", atol_scale=5e-5)


# ---- 5. in-place updates and non-leaf values ------------------------------------------------------------------------
def test_inplace_update_and_non_leaf_values():
    B, N, C, Din, h, Ks, Kc = 2, 48, 4, 3, 8, 3, 2
    rowptr, col, vals = pattern(N, 6, seed=6, zero_frac=0.0)
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=6)
    args = [t[k].float().to(DEV) for k in ARGS]
    dHn = t["dHn"].float().to(DEV)
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc)
    ps, v = learnable_partition(rowptr, col, vals, N, 0, 1)
    S.halo.partitioned_cell_forward(ps, *args, Ks, Kc).backward(dHn)
    with torch.no_grad():                                              # one SGD step, in place
        v.sub_(0.5 * v.grad / v.grad.abs().max() * v.abs().max())
    v.grad = None
    Hn = S.halo.partitioned_cell_forward(ps, *args, Ks, Kc)
    Hn.backward(dHn)
    torch.cuda.synchronize()
    t["Gs"] = dense_of(rowptr, col, v.detach().cpu(), N)
    Hn_o, g_o = oracle_cell_with_grads(t, cfg)
    O.assert_close(Hn.detach().cpu(), Hn_o, "H' after the update")
    O.assert_close(v.grad.cpu(), g_o["dGs"][edge_rows(rowptr), col.long()], "dvals after the update")
    # autograd refuses a backward after an in-place change of the values
    Hn = S.halo.partitioned_cell_forward(ps, *args, Ks, Kc)
    with torch.no_grad():
        v.mul_(1.5)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        Hn.backward(dHn)
    # non-leaf values: softplus(raw) through with_values, the gradient reaches raw
    raw0 = torch.log(torch.expm1(vals.double())).float()               # softplus(raw0) == vals
    raw = torch.nn.Parameter(raw0.to(DEV))
    psv = ps.with_values(torch.nn.functional.softplus(raw))
    assert psv.fwd is ps.fwd and psv.vals is not ps.vals
    Hn = S.halo.partitioned_cell_forward(psv, *args, Ks, Kc)
    Hn.backward(dHn)
    torch.cuda.synchronize()
    t["Gs"] = dense_of(rowptr, col, torch.nn.functional.softplus(raw0.double()), N)
    Hn_o, g_o = oracle_cell_with_grads(t, cfg)
    O.assert_close(Hn.detach().cpu(), Hn_o, "H' with_values")
    O.assert_close(raw.grad.cpu(), g_o["dGs"][edge_rows(rowptr), col.long()] * torch.sigmoid(raw0.double()), "d raw")


# ---- 6. a constant partitioned support never launches the gradient variant ------------------------------------------
def test_constant_partitioned_support_launches_no_gradient_hop():
    from stc_gnn_b200 import _lib
    B, N, C, Din, h, Ks, Kc = 2, 64, 4, 3, 8, 3, 2
    rowptr, col, vals = pattern(N, 6, seed=8)
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=8)

    def kinds_of(ps):
        args = [t[k].float().to(DEV).requires_grad_(True) for k in ARGS]
        _lib.timing_enable(True)
        _lib.timing_collect()
        S.halo.partitioned_cell_forward(ps, *args, Ks, Kc).backward(t["dHn"].float().to(DEV))
        torch.cuda.synchronize()
        _lib.timing_enable(False)
        return _lib.timing_collect()

    const = kinds_of(S.halo.PartitionedSupport(rowptr, col, vals, N, 0, 1))
    assert "support_csr_grad" not in const and const["support_csr"][1] > 0, const
    learned = kinds_of(learnable_partition(rowptr, col, vals, N, 0, 1)[0])
    assert learned["support_csr_grad"][1] == 3 * (Ks - 1), learned   # every adjoint hop of the three chains


# ---- 7. two ranks ------------------------------------------------------------------------------------------------------
def _two_rank_worker(rank, world, port, backend, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        dev = torch.device("cuda", rank if backend == "nccl" else 0)
        torch.cuda.set_device(dev)
        if backend == "nccl":
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        else:
            dist.init_process_group("gloo", rank=rank, world_size=world)
        for shape in ((2, 101, 5, 16, 16, 3, 2), (1, 64, 4, 1, 8, 4, 2)):
            ps = _learned_cell_block(rank, world, dev, shape, seed=33, check_ranks_agree=True)
            assert ps.fwd.nhalo > 0
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, None))
    except Exception:  # pragma: no cover - reported by the parent
        q.put((rank, traceback.format_exc()))


def _run_two_ranks(backend):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, backend, q)) for r in range(2)]
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
def test_learnable_halo_cell_two_ranks_nccl():
    _run_two_ranks("nccl")


def test_learnable_halo_cell_two_ranks_gloo_one_gpu():
    """Both ranks on one GPU, exchanging over gloo (its CUDA all-to-all) from hop_ext's side stream."""
    _run_two_ranks("gloo")
