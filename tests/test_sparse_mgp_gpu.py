"""The graph generator on a fixed CSR pattern on the GPU (stc_pair_scores_csr, stc_edge_softmax_fwd / _bwd,
`pair_softmax_csr`, `SparseGraphGenerator`): the kernels against the fp64 restatement (tests/sparse_mgp_oracle.py) and
their determinism, the complete pattern against the dense generator, the config 3 grid, a generator feeding a
RecurrentStack, peak memory, the no-grad path, two-rank batch data-parallelism and the error paths.

Tolerance: |got - ref| <= 1e-4 * |ref| + 1e-5 * mean|ref|.  Two wider floors, each stated where it is used: 5e-5 *
mean|ref| for the Wu / Wv gradients of the generator (the fp32 torch dense generator's own worst error on the
complete-pattern inputs below is 0.9-1.2e-5 * mean|ref| against fp64, and at another seed of the same shape one of its
elements falls outside the 1e-5 floor) and 5e-5 through a stack, as in the other stack tests.  Inputs are chosen so
that no stored edge other than a self-loop has |S| < 1e-3 * mean|S| (asserted): a relu boundary flip between fp32 and
fp64 then cannot decide a comparison."""
import os
import socket
import traceback

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from stc_gnn_b200 import _lib, dp, mgp
from stc_gnn_b200.sparse_mgp import _EdgeSoftmax, _PairScores
from stc_gnn_b200.synth import grid_csr, knn_csr
from tests import sparse_mgp_oracle as SO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GEN_FLOOR = 5e-5     # Wu / Wv gradients of the generator (module docstring)
STACK_FLOOR = 5e-5


def csr(rowptr, col, dev=DEV):
    """A pattern whose stored values (some explicit zeros) the generator must ignore."""
    vals = torch.rand(col.numel(), generator=torch.Generator().manual_seed(0))
    vals[::5] = 0.0
    return S.CsrSupport(rowptr.to(dev), col.to(dev), vals.to(dev), rowptr.numel() - 1)


def assert_margin(S64, rowptr, col):
    loops = SO.edge_rows(rowptr) == col.long()
    small = (S64.abs() < 1e-3 * S64.abs().mean()) & ~loops
    assert not small.any(), f"{int(small.sum())} stored edges score within 1e-3 * mean|S| of 0"


def safe(rowptr, col, U64, V64):
    """The pattern without the few edges whose fp64 score is within 1e-3 * mean|S| of 0 (self-loops stay)."""
    S64 = SO.pair_scores_at(U64, V64, rowptr, col)
    rowptr, col, _ = SO.drop_near_zero_scores(rowptr, col, S64)
    assert_margin(SO.pair_scores_at(U64, V64, rowptr, col), rowptr, col)
    return rowptr, col


# ---- 1. the kernels on their own ------------------------------------------------------------------------------------
def _kernel_pass(U, V, pat, w):
    Ul, Vl = U.clone().requires_grad_(True), V.clone().requires_grad_(True)
    Sc = _PairScores.apply(Ul, Vl, pat)
    Sc.retain_grad()
    P = _EdgeSoftmax.apply(Sc, pat)
    (P * w).sum().backward()
    torch.cuda.synchronize()
    return Sc.detach(), P.detach(), Sc.grad, Ul.grad, Vl.grad


@pytest.mark.parametrize("width", [1, 3, 4, 384, 1100])
def test_kernels_against_fp64_and_bitwise_repeatable(width):
    """Widths 1 / 3 take the scalar path, 4 / 384 / 1100 the 16-byte path; 1100 spans three 512-float chunks (and the
    scalar path sweeps 128 floats a chunk).  The pattern has empty rows, self-loops, is asymmetric, and row 40 stores
    more than 64 edges."""
    N = 300
    g = torch.Generator().manual_seed(width)
    U = torch.randn(N, width, generator=g) * width ** -0.25     # |S| of order 1 at every width
    V = torch.randn(N, width, generator=g) * width ** -0.25
    rowptr, col = SO.random_pattern(N, 9, seed=width, empty_every=7, hub=(40, 120))
    rowptr, col = safe(rowptr, col, U.double(), V.double())
    assert int(rowptr[41] - rowptr[40]) > 64 and (rowptr[1:] == rowptr[:-1]).any()
    pat = csr(rowptr, col)
    w = torch.randn(col.numel(), generator=g)

    got = _kernel_pass(U.to(DEV), V.to(DEV), pat, w.to(DEV))
    again = _kernel_pass(U.to(DEV), V.to(DEV), pat, w.to(DEV))
    for name, a, b in zip(("S", "P", "dS", "dU", "dV"), got, again):
        assert torch.equal(a, b), f"{name} differs between two calls"

    U64, V64 = U.double().requires_grad_(True), V.double().requires_grad_(True)
    S64 = SO.pair_scores_at(U64, V64, rowptr, col)
    S64.retain_grad()
    P64 = SO.edge_softmax(S64, rowptr)
    (P64 * w.double()).sum().backward()
    loops = (SO.edge_rows(rowptr) == col.long()).to(DEV)
    assert loops.any() and torch.all(got[0][loops] == 0.0), "a self-loop must score exactly 0"
    for name, a, b in zip(("S", "P", "dS", "dU", "dV"), got, (S64, P64, S64.grad, U64.grad, V64.grad)):
        O.assert_close(a.cpu(), b.detach(), f"{name} (width {width})")


# ---- 2. complete pattern at the SF shape: the dense generator -------------------------------------------------------
def test_complete_pattern_is_the_dense_generator():
    B, T, N, C, hg, seed = 4, 12, 100, 5, 16, 133
    g = torch.Generator().manual_seed(seed)
    X = (torch.rand(B, T, N, C, generator=g) < 0.3).float()                        # incident flags, as in the SF data
    torch.manual_seed(seed)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    w = torch.randn(N, N, generator=g)
    Wu64 = gen.params_S["Wu"].detach().double().cpu().requires_grad_(True)
    Wv64 = gen.params_S["Wv"].detach().double().cpu().requires_grad_(True)
    Sd = mgp.pair_scores(X.double(), Wu64, Wv64, gen.alpha)
    rowptr, col = SO.complete_pattern(N)
    assert_margin(Sd.detach().reshape(-1), rowptr, col)
    P64 = torch.softmax(torch.relu(Sd), -1)
    (P64 * w.double()).sum().backward()

    sup = gen(X.to(DEV), csr(rowptr, col))
    assert sup.learnable
    (sup.vals * w.reshape(-1).to(DEV)).sum().backward()
    O.assert_close(sup.vals.detach().cpu().reshape(N, N), P64.detach(), "P vs the dense generator")
    O.assert_close(gen.params_S["Wu"].grad.cpu(), Wu64.grad, "dWu", atol_scale=GEN_FLOOR)
    O.assert_close(gen.params_S["Wv"].grad.cpu(), Wv64.grad, "dWv", atol_scale=GEN_FLOOR)


# ---- 3. the config 3 grid -------------------------------------------------------------------------------------------
def test_grid_generator_against_fp64():
    B, T, C, hg = 2, 3, 4, 8
    rowptr, col, _ = grid_csr(64, 64)
    N = 4096
    g = torch.Generator().manual_seed(3)
    X = torch.randn(B, T, N, C, generator=g)
    torch.manual_seed(3)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    Wu64 = gen.params_S["Wu"].detach().double().cpu().requires_grad_(True)
    Wv64 = gen.params_S["Wv"].detach().double().cpu().requires_grad_(True)
    X64 = X.double().requires_grad_(True)
    with torch.no_grad():
        rowptr, col = safe(rowptr, col, SO.node_major(X64, Wu64, gen.alpha), SO.node_major(X64, Wv64, gen.alpha))
    w = torch.randn(col.numel(), generator=g)
    P64 = SO.sparse_generator(X64, Wu64, Wv64, gen.alpha, rowptr, col)
    (P64 * w.double()).sum().backward()

    Xd = X.to(DEV).requires_grad_(True)
    sup = gen(Xd, csr(rowptr, col))
    (sup.vals * w.to(DEV)).sum().backward()
    O.assert_close(sup.vals.detach().cpu(), P64.detach(), "P (grid)")
    O.assert_close(gen.params_S["Wu"].grad.cpu(), Wu64.grad, "dWu (grid)", atol_scale=GEN_FLOOR)
    O.assert_close(gen.params_S["Wv"].grad.cpu(), Wv64.grad, "dWv (grid)", atol_scale=GEN_FLOOR)
    O.assert_close(Xd.grad.cpu(), X64.grad, "dX_seq (grid)")


# ---- 4. generator -> RecurrentStack -> loss -> backward ----------------------------------------------------------------
@pytest.mark.parametrize("Ks", [2, 3])
def test_generator_feeds_a_stack(Ks):
    N, C, Kc, h, layers, horizon, B, T, hg = 48, 3, 2, 8, 2, 2, 2, 3, 4
    g = torch.Generator().manual_seed(40 + Ks)
    X = torch.randn(B, T, N, C, generator=g)
    torch.manual_seed(40 + Ks)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    stack = S.RecurrentStack(N, C, Ks, Kc, 1, h, layers, horizon).to(DEV)
    Gc = (torch.rand(C, C, generator=g) / C)
    dOut = torch.randn(B, horizon, N, C, h, generator=g)
    Wu64 = gen.params_S["Wu"].detach().double().cpu().requires_grad_(True)
    Wv64 = gen.params_S["Wv"].detach().double().cpu().requires_grad_(True)
    rowptr, col = SO.random_pattern(N, 6, seed=Ks, empty_every=9)
    rowptr, col = safe(rowptr, col, SO.node_major(X.double(), Wu64.detach(), gen.alpha),
                       SO.node_major(X.double(), Wv64.detach(), gen.alpha))

    out = stack(gen(X.to(DEV), csr(rowptr, col)), Gc.to(DEV), X.to(DEV)[..., None])
    out.backward(dOut.to(DEV))
    torch.cuda.synchronize()

    P64 = SO.sparse_generator(X.double(), Wu64, Wv64, gen.alpha, rowptr, col)
    Gs64 = SO.dense_of(rowptr, col, P64, N)
    cp = lambda c: O.CellParams(c.gates.W.detach().double().cpu(), c.gates.b.detach().double().cpu(),
                                c.candi.W.detach().double().cpu(), c.candi.b.detach().double().cpu())
    ref = O.stack_forward(Gs64, Gc.double(), X.double()[..., None], [cp(c) for c in stack.encoder],
                          [cp(c) for c in stack.decoder], horizon, Ks, Kc)
    ref.backward(dOut.double())
    O.assert_close(out.detach().cpu(), ref.detach(), f"stack output (Ks {Ks})", atol_scale=STACK_FLOOR)
    O.assert_close(gen.params_S["Wu"].grad.cpu(), Wu64.grad, f"dWu through the stack (Ks {Ks})", atol_scale=STACK_FLOOR)
    O.assert_close(gen.params_S["Wv"].grad.cpu(), Wv64.grad, f"dWv through the stack (Ks {Ks})", atol_scale=STACK_FLOOR)


# ---- 5. memory: no per-edge slab ---------------------------------------------------------------------------------------
def test_peak_memory_has_no_per_edge_slab():
    """kNN N = 65,536 (8 or more edges a row), B = 2, T = 12, C = 8, hg = 16: width 384, so one gathered [nnz, width]
    operand of the per-edge torch form is 0.93 GB and its four operands 3.7 GB.  The generator's forward + backward
    stays below about a dozen node-sized tensors."""
    B, T, C, hg = 2, 12, 8, 16
    rowptr, col, _ = knn_csr(65536, 8)
    N, nnz, width = 65536, col.numel(), B * T * hg
    assert int((rowptr[1:] - rowptr[:-1]).min()) >= 8 and 4 * nnz * width > 256e6
    pat = csr(rowptr, col)
    X = torch.randn(B, T, N, C, device=DEV)
    torch.manual_seed(0)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    w = torch.randn(nnz, device=DEV)
    (gen(X, pat).vals * w).sum().backward()               # warm: the pattern's transpose permutation is built once
    gen.zero_grad(set_to_none=False)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    (gen(X, pat).vals * w).sum().backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    bound = 12 * 4 * N * width + 64 * nnz
    assert peak < bound, (peak, bound, 4 * 4 * nnz * width)


# ---- 6. no_grad: a constant support ---------------------------------------------------------------------------------
def test_no_grad_gives_a_constant_support():
    B, T, N, C, hg, h, Ks, Kc = 2, 3, 64, 3, 4, 8, 3, 2
    g = torch.Generator().manual_seed(6)
    X = torch.randn(B, T, N, C, generator=g).to(DEV)
    torch.manual_seed(6)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    rowptr, col = SO.random_pattern(N, 6, seed=6)
    pat = csr(rowptr, col)
    with torch.no_grad():
        sup = gen(X, pat)
    assert not sup.learnable and not sup.vals.requires_grad
    with_grad = gen(X, pat)
    assert torch.equal(sup.vals, with_grad.vals.detach())
    cell = S.STC_Cell(N, C, Ks, Kc, 1, h).to(DEV)
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
    assert gen.params_S["Wu"].grad is None


# ---- 7. error paths --------------------------------------------------------------------------------------------------
def test_error_paths():
    gen = S.SparseGraphGenerator(4, 8).to(DEV)
    rowptr, col = SO.random_pattern(20, 4, seed=1)
    pat = csr(rowptr, col)
    X = torch.randn(2, 3, 20, 4, device=DEV)
    with pytest.raises(RuntimeError, match="no CPU path"):
        gen(X.cpu(), pat)
    with pytest.raises(RuntimeError, match="20 nodes, the input 21"):
        gen(torch.randn(2, 3, 21, 4, device=DEV), pat)
    with pytest.raises(RuntimeError, match="5 categories"):
        gen(torch.randn(2, 3, 20, 5, device=DEV), pat)
    with pytest.raises(RuntimeError, match="CsrSupport"):
        gen(X, torch.zeros(20, 20, device=DEV))
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.pair_softmax_csr(torch.zeros(20, 6), torch.zeros(20, 6), pat)
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    bad = S.support.dense_struct(torch.zeros(20, 20, device=DEV))
    U = torch.zeros(20, 6, device=DEV)
    assert lib.stc_pair_scores_csr(bad, 20, 6, U.data_ptr(), U.data_ptr(), U.data_ptr(), st) == -2
    assert b"CSR" in lib.stc_last_error()
    assert lib.stc_pair_scores_csr(pat.struct(), 20, 0, U.data_ptr(), U.data_ptr(), U.data_ptr(), st) == -1
    assert lib.stc_edge_softmax_fwd(pat.struct(), 0, U.data_ptr(), U.data_ptr(), st) == -1
    assert lib.stc_edge_softmax_bwd(pat.struct(), 20, U.data_ptr(), None, U.data_ptr(), U.data_ptr(), st) == -1


# ---- 8. batch data-parallel, two ranks ---------------------------------------------------------------------------------
def _dp_case(rank, world, dev):
    """Each rank holds a shard of the batch.  The shard P equals the single-process global-batch P, and after the
    bucket all-reduce the Wu / Wv gradients equal the global-batch ones, for a summed (average=False) and an averaged
    (average=True) bucket.  The global-batch run uses a one-rank group, i.e. no communication."""
    B, T, N, C, hg = 4, 3, 80, 3, 6
    singles = [dist.new_group([r]) for r in range(world)]
    g = torch.Generator().manual_seed(9)
    X = torch.randn(B, T, N, C, generator=g)
    torch.manual_seed(9)
    gen = S.SparseGraphGenerator(C, hg).to(dev)
    rowptr, col = SO.random_pattern(N, 7, seed=9, empty_every=6)
    with torch.no_grad():
        rowptr, col = safe(rowptr, col, SO.node_major(X.double(), gen.params_S["Wu"].double().cpu(), gen.alpha),
                           SO.node_major(X.double(), gen.params_S["Wv"].double().cpu(), gen.alpha))
    pat = csr(rowptr, col, dev)
    wS = torch.randn(B, col.numel(), generator=g).to(dev)        # per-sample loss weights
    sl = slice(*dp.shard_bounds(B, rank, world))
    Xd = X.to(dev)
    for average in (False, True):
        gen.zero_grad(set_to_none=True)
        P_full = gen(Xd, pat, group=singles[rank]).vals
        ((P_full * wS.sum(0)).sum() / (world if average else 1)).backward()
        full = [p.grad.clone() for p in gen.parameters()]
        gen.zero_grad(set_to_none=True)
        P_r = gen(Xd[sl], pat, average=average).vals
        O.assert_close(P_r.detach().cpu(), P_full.detach().cpu(), f"shard P (rank {rank})")
        (P_r * wS[sl].sum(0)).sum().backward()
        for p in gen.parameters():
            dist.all_reduce(p.grad)
            if average:
                p.grad.div_(world)
        for (n, p), want in zip(gen.named_parameters(), full):
            O.assert_close(p.grad.cpu(), want.cpu(), f"d{n} (rank {rank}, average={average})", atol_scale=GEN_FLOOR)


def _two_rank_worker(rank, world, port, backend, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        dev = torch.device("cuda", rank if backend == "nccl" else 0)
        torch.cuda.set_device(dev)
        if backend == "nccl":
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        else:
            dist.init_process_group("gloo", rank=rank, world_size=world)
        _dp_case(rank, world, dev)
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
def test_generator_batch_dp_two_ranks_nccl():
    _run_two_ranks("nccl")


def test_generator_batch_dp_two_ranks_gloo_one_gpu():
    _run_two_ranks("gloo")
