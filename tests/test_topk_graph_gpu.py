"""The sparse generator choosing its own pattern on the GPU (stc_pair_topk, `pair_topk`, `topk_pattern`,
`SparseGraphGenerator(..)(X_seq, k=k)`): the selection against the fp64 oracle (tests/topk_graph_oracle.py) at small
shapes and at the config 4 size, determinism, the generator on the selected pattern, a generated support feeding a
RecurrentStack, the no-grad path, no host synchronisation, peak memory and the error paths.

Selection margin: with t the fp64 k-th score of a row and tau = 1e-5 max|S_row|, every column with S > t + tau must be
selected and none with S < t - tau (3xTF32 scores carry about 1e-6 relative error).  Values: 1e-4 |ref| + 1e-5
mean|ref|; the Wu / Wv gradients and the stack take the 5e-5 floors of tests/test_sparse_mgp_gpu.py."""
import pytest
import torch

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from stc_gnn_b200 import _lib, mgp
from stc_gnn_b200.halo import PartitionedSupport
from tests import sparse_mgp_oracle as SO
from tests import topk_graph_oracle as TO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GEN_FLOOR = 5e-5
STACK_FLOOR = 5e-5


def uv(N, W, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.tanh(torch.randn(N, W, generator=g)).to(DEV), torch.tanh(torch.randn(N, W, generator=g)).to(DEV))


def check_scores(got, S64, cols, what):
    ref = S64.gather(1, cols.long())
    O.assert_close(got.double().cpu(), ref.cpu(), what)
    diag = cols.long() == torch.arange(cols.shape[0], device=cols.device)[:, None]
    assert torch.all(got[diag] == 0), f"{what}: a selected diagonal entry is not exactly 0"


# ---- 1. the selection against fp64 -----------------------------------------------------------------------------------
@pytest.mark.parametrize("W", [4, 36, 384, 1536])
@pytest.mark.parametrize("N", [1, 7, 100, 128, 129, 300, 1000, 4096])
def test_selection_against_fp64(N, W):
    """W % 32 != 0 (4, 36) ends the K halves on partial atoms; N = 129 / 300 / 1000 leave partial row blocks and column
    tiles, N = 4096 splits the columns into segments."""
    U, V = uv(N, W, 1000 * N + W)
    S64 = TO.full_scores(U.double(), V.double())
    near = 0
    for k in (1, 8, 16, 32):
        if k > N:
            continue
        cols, sc = S.pair_topk(U, V, k, scores=True)
        near += TO.check_selection(S64, cols, k)
        check_scores(sc, S64, cols, f"scores (N {N}, W {W}, k {k})")
        cols2, sc2 = S.pair_topk(U, V, k, scores=True)
        assert torch.equal(cols, cols2) and torch.equal(sc, sc2), "two calls differ"
        assert torch.equal(S.pair_topk(U, V, k), cols)
    print(f"N {N} W {W}: {near} near-tie rows")


def test_ties_go_to_the_smaller_column():
    """Rows 0..7 of U / V repeat as rows 8..15 etc. (N = 64), so columns m, m + 8, m + 16, ... of a row have the same
    operand rows and bitwise the same score (except the family of the diagonal, whose member n is forced to 0).  Of such
    a family the selection must take the smaller columns first."""
    U, V = uv(8, 32, 7)
    U, V = U.repeat(8, 1), V.repeat(8, 1)
    S64 = TO.full_scores(U.double(), V.double())
    for k in (1, 5, 16, 32):
        cols = S.pair_topk(U, V, k).cpu()
        TO.check_selection(S64, cols, k)
        for n in range(64):
            chosen = set(cols[n].tolist())
            for m in chosen:
                if m % 8 != n % 8:
                    assert all(m2 in chosen for m2 in range(m % 8, m, 8)), (n, k, sorted(chosen))


def test_nan_and_inf_rows_still_select_valid_columns():
    """A NaN (missing data, a diverging run) or an inf in one node's row makes that row's and that column's scores NaN.
    They rank as -inf: the NaN row keeps its diagonal (score 0) and then the smallest columns, every other row never
    selects the NaN column unless it must, and all columns lie in [0, N) and ascend.  The same through the generator: the
    selected pattern is valid and P is what the fixed-pattern path gives on it."""
    N, W = 300, 36
    for bad in (float("nan"), float("inf")):
        U, V = uv(N, W, 11)
        U[17, 5] = bad
        for k in (1, 8, 32):
            cols, sc = S.pair_topk(U, V, k, scores=True)
            torch.cuda.synchronize()
            c = cols.long().cpu()
            assert int(c.min()) >= 0 and int(c.max()) < N and torch.all(c[:, 1:] > c[:, :-1]), (bad, k)
            want = sorted(([17] + [m for m in range(N) if m != 17][:k - 1]))
            assert c[17].tolist() == want, (bad, k, c[17].tolist())
            assert not (c == 17).any(1)[torch.arange(N) != 17].any(), (bad, k)
            keep = torch.arange(N, device=DEV) != 17
            S64 = TO.full_scores(U.double(), V.double())
            S64[:, 17] = S64[keep][:, keep].min() - 1.0   # ranks last, and keeps the margin tau finite
            keep = torch.arange(N, device=DEV) != 17
            TO.check_selection(S64[keep], cols[keep], k)
    X = torch.randn(2, 3, N, 4, device=DEV)
    X[1, 2, 40, 0] = float("nan")
    gen = S.SparseGraphGenerator(4, 8).to(DEV)
    sup = gen(X, k=8)
    torch.cuda.synchronize()
    assert int(sup.col.min()) >= 0 and int(sup.col.max()) < N
    fixed = S.CsrSupport(sup.rowptr, sup.col, torch.ones(N * 8, device=DEV), N)
    assert torch.equal(gen(X, fixed).vals.nan_to_num(), sup.vals.nan_to_num())


def test_full_size_config4():
    """N = 65,536, width 384 (B = 2, T = 12, hg = 16): one segment of 512 column tiles a row block.  256 sampled rows
    against fp64 scores over all 65,536 columns, and bitwise determinism."""
    N, W, k = 65536, 384, 32
    U, V = uv(N, W, 4)
    cols, sc = S.pair_topk(U, V, k, scores=True)
    cols2, sc2 = S.pair_topk(U, V, k, scores=True)
    assert torch.equal(cols, cols2) and torch.equal(sc, sc2)
    rows = torch.randperm(N, generator=torch.Generator().manual_seed(0))[:256].to(DEV)
    S64 = TO.full_scores(U.double(), V.double(), rows)
    near = TO.check_selection(S64, cols[rows], k)
    check_scores(sc[rows], S64, cols[rows], "scores (config 4)")
    print(f"config 4: {near} near-tie rows of 256")


def test_peak_memory_is_the_workspace_and_the_outputs():
    N, W, k = 65536, 384, 16
    U, V = uv(N, W, 5)
    ws = _lib.load().stc_pair_topk_workspace_bytes(N, W, k)
    S.pair_topk(U, V, k)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    S.pair_topk(U, V, k, scores=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak <= ws + 8 * N * k + (1 << 20), (peak, ws)
    assert peak < 4 * N * N / 100


# ---- 2. the generator on the selected pattern --------------------------------------------------------------------------
def _assert_margin(P_scores, cols):
    """no selected edge other than a self-loop scores within 1e-3 * mean|S| of 0 (a relu flip would decide a gradient)"""
    diag = cols.long() == torch.arange(cols.shape[0])[:, None]
    small = (P_scores.abs() < 1e-3 * P_scores.abs().mean()) & ~diag
    assert not small.any(), f"{int(small.sum())} selected edges score within 1e-3 * mean|S| of 0"


@pytest.mark.parametrize("N,k", [(300, 8), (1000, 32)])
def test_generator_selects_then_generates(N, k):
    B, T, C, hg = 2, 3, 4, 8
    g = torch.Generator().manual_seed(N + k)
    X = torch.randn(B, T, N, C, generator=g)
    torch.manual_seed(N)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    w = torch.randn(N * k, generator=g)
    Xd = X.to(DEV).requires_grad_(True)
    sup = gen(Xd, k=k)
    assert sup.learnable and sup.nnz == N * k and torch.equal(sup.rowptr.cpu(), (torch.arange(N + 1) * k).int())
    (sup.vals * w.to(DEV)).sum().backward()
    # the same P on the fixed pattern it selected, bitwise
    fixed = S.CsrSupport(sup.rowptr, sup.col, torch.ones(N * k, device=DEV), N)
    assert torch.equal(gen(X.to(DEV), fixed).vals, sup.vals)
    cols = sup.col.reshape(N, k).cpu()
    Wu64 = gen.params_S["Wu"].detach().double().cpu().requires_grad_(True)
    Wv64 = gen.params_S["Wv"].detach().double().cpu().requires_grad_(True)
    X64 = X.double().requires_grad_(True)
    with torch.no_grad():
        U64, V64 = SO.node_major(X64, Wu64, gen.alpha), SO.node_major(X64, Wv64, gen.alpha)
        S64 = TO.full_scores(U64, V64)
        TO.check_selection(S64, cols, k)
        _assert_margin(S64.gather(1, cols.long()), cols)
    rowptr = sup.rowptr.cpu()
    P64 = SO.sparse_generator(X64, Wu64, Wv64, gen.alpha, rowptr, cols.reshape(-1))
    (P64 * w.double()).sum().backward()
    O.assert_close(sup.vals.detach().cpu(), P64.detach(), "P (selected)")
    O.assert_close(gen.params_S["Wu"].grad.cpu(), Wu64.grad, "dWu (selected)", atol_scale=GEN_FLOOR)
    O.assert_close(gen.params_S["Wv"].grad.cpu(), Wv64.grad, "dWv (selected)", atol_scale=GEN_FLOOR)
    O.assert_close(Xd.grad.cpu(), X64.grad, "dX_seq (selected)")


@pytest.mark.parametrize("N", [5, 32])
def test_k_equal_n_is_the_dense_generator(N):
    B, T, C, hg = 2, 4, 3, 6
    g = torch.Generator().manual_seed(N)
    X = torch.randn(B, T, N, C, generator=g)
    torch.manual_seed(N)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    sup = gen(X.to(DEV), k=N)
    assert torch.equal(sup.col.cpu(), torch.arange(N, dtype=torch.int32).repeat(N))
    Wu, Wv = gen.params_S["Wu"].detach().double().cpu(), gen.params_S["Wv"].detach().double().cpu()
    Ps = torch.softmax(torch.relu(mgp.pair_scores(X.double(), Wu, Wv, gen.alpha)), -1)
    O.assert_close(sup.vals.detach().cpu().reshape(N, N), Ps, f"k = N = {N} vs the dense generator")


@pytest.mark.parametrize("Ks", [2, 4])
def test_generated_support_feeds_a_stack(Ks):
    N, C, Kc, h, layers, horizon, B, T, hg, k = 64, 3, 2, 8, 2, 2, 2, 3, 4, 6
    g = torch.Generator().manual_seed(50 + Ks)
    X = torch.randn(B, T, N, C, generator=g)
    torch.manual_seed(50 + Ks)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    stack = S.RecurrentStack(N, C, Ks, Kc, 1, h, layers, horizon).to(DEV)
    Gc = torch.rand(C, C, generator=g) / C
    dOut = torch.randn(B, horizon, N, C, h, generator=g)
    sup = gen(X.to(DEV), k=k)
    out = stack(sup, Gc.to(DEV), X.to(DEV)[..., None])
    out.backward(dOut.to(DEV))
    torch.cuda.synchronize()

    Wu64 = gen.params_S["Wu"].detach().double().cpu().requires_grad_(True)
    Wv64 = gen.params_S["Wv"].detach().double().cpu().requires_grad_(True)
    rowptr, col = sup.rowptr.cpu(), sup.col.cpu()
    with torch.no_grad():
        S64 = TO.full_scores(SO.node_major(X.double(), Wu64, gen.alpha), SO.node_major(X.double(), Wv64, gen.alpha))
        TO.check_selection(S64, col.reshape(N, k), k)
        _assert_margin(S64.gather(1, col.reshape(N, k).long()), col.reshape(N, k))
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


def test_no_grad_gives_a_constant_support():
    X = torch.randn(2, 3, 64, 3, device=DEV)
    gen = S.SparseGraphGenerator(3, 4).to(DEV)
    with torch.no_grad():
        sup = gen(X, k=8)
    assert not sup.learnable and not sup.vals.requires_grad
    assert torch.equal(sup.vals, gen(X, k=8).vals.detach())


def test_forward_makes_no_host_synchronisation():
    B, T, N, C, hg, k = 2, 12, 4096, 8, 16, 16
    X = torch.randn(B, T, N, C, device=DEV)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    gen(X, k=k)                                   # warm: library load, allocator, kernels
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        sup = gen(X, k=k)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert sup.learnable and sup.nnz == N * k


def test_timing_kind():
    U, V = uv(512, 64, 9)
    _lib.timing_enable(True)
    _lib.timing_collect()
    S.pair_topk(U, V, 8)
    torch.cuda.synchronize()
    _lib.timing_enable(False)
    kinds = _lib.timing_collect()
    assert kinds["pair_topk"][1] == 1 and kinds["pair_topk"][2] == 8.0 * 512 * 64 + 8.0 * 512 * 8, kinds


# ---- 3. error paths ------------------------------------------------------------------------------------------------------
def test_error_paths():
    U = torch.zeros(20, 6, device=DEV)
    for bad in (0, -1, 33, 21):
        with pytest.raises(RuntimeError, match=f"k = {bad} outside"):
            S.pair_topk(U, U, bad)
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.pair_topk(U.cpu(), U.cpu(), 4)
    with pytest.raises(RuntimeError, match="float32"):
        S.pair_topk(U.double(), U.double(), 4)
    gen = S.SparseGraphGenerator(4, 8).to(DEV)
    X = torch.randn(2, 3, 20, 4, device=DEV)
    pat = S.CsrSupport(torch.arange(21, dtype=torch.int32, device=DEV), torch.arange(20, dtype=torch.int32, device=DEV),
                       torch.ones(20, device=DEV), 20)
    with pytest.raises(RuntimeError, match="exactly one of `pattern`"):
        gen(X, pat, k=4)
    with pytest.raises(RuntimeError, match="exactly one of `pattern`"):
        gen(X)
    with pytest.raises(RuntimeError, match="row-partitioned"):
        gen(X, PartitionedSupport.__new__(PartitionedSupport), k=4)
    with pytest.raises(RuntimeError, match="batch data-parallelism"):
        gen(X, k=4, group=object())
    for bad in (0, 33, 21):
        with pytest.raises(RuntimeError, match=f"k = {bad} outside"):
            gen(X, k=bad)
    with pytest.raises(RuntimeError, match="no CPU path"):
        gen(X.cpu(), k=4)
    # the C ABI: every check returns before a launch
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    cols = torch.empty(20, 32, dtype=torch.int32, device=DEV)
    ws = torch.empty(1 << 20, dtype=torch.uint8, device=DEV)
    U8 = torch.zeros(20, 8, device=DEV)
    args = lambda k, width=8, nbytes=1 << 20: (20, width, U8.data_ptr(), U8.data_ptr(), k, cols.data_ptr(), None,
                                               ws.data_ptr(), nbytes, st)
    assert lib.stc_pair_topk(*args(33)) == -2 and b"at most 32" in lib.stc_last_error()
    assert lib.stc_pair_topk(*args(0)) == -1
    assert lib.stc_pair_topk(*args(21)) == -1
    assert lib.stc_pair_topk(*args(4, width=6)) == -1
    assert lib.stc_pair_topk(*args(4, nbytes=16)) == -3
    assert lib.stc_pair_topk_workspace_bytes(20, 8, 33) == 0 and lib.stc_pair_topk_workspace_bytes(20, 6, 4) == 0
    assert lib.stc_pair_topk(*args(4)) == 0
    torch.cuda.synchronize()
