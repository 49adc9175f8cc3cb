"""Bitwise-repeatable gradients under torch.use_deterministic_algorithms(True).  Each case runs forward + backward three
times from fresh .grad -- once with an unrelated matmul running on another stream, so that CTA scheduling differs --
and requires every output and gradient to be bitwise equal across the runs and within the fp64-oracle tolerance.
The fixed-order reduction kernel (det_reduce) must run in this mode and not in the default one."""
import pytest
import torch

import stc_gnn_b200 as S
from oracle import stc_oracle as O
from stc_gnn_b200 import _lib
from tests.helpers import oracle_cell_with_grads, random_case

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


@pytest.fixture
def deterministic():
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(was)
    _lib.sync_deterministic()
    _lib.set_concurrency(-1)


def _busy_stream():
    """A large matmul on another stream, enqueued right before the step: it holds SMs while the step's kernels start."""
    s = torch.cuda.Stream()
    a = torch.randn(8192, 8192, device=DEV)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for _ in range(4):
            a = a @ a * 1e-4
    return s, a


def repeat3(step):
    """step() -> dict of tensors; three runs, the second beside a busy stream; returns the first run's results."""
    runs = []
    for i in range(3):
        busy = _busy_stream() if i == 1 else None
        out = step()
        torch.cuda.synchronize()
        runs.append({k: v.detach().clone() for k, v in out.items() if v is not None})
        del busy
    for k in runs[0]:
        for r in runs[1:]:
            assert torch.equal(runs[0][k], r[k]), f"{k} differs between two deterministic runs"
    return runs[0]


def kinds_of(step):
    _lib.timing_enable(True)
    _lib.timing_collect()
    step()
    torch.cuda.synchronize()
    _lib.timing_enable(False)
    return {k for k, v in _lib.timing_collect().items() if v[1]}


def cell_case(shape, support="dense", seed=0, concurrency=-1):
    B, N, C, Din, h, Ks, Kc = shape
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=seed, sparse_frac=0.8 if support != "dense" else None)
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, activation=None)
    leaf = lambda k: t[k].float().to(DEV).requires_grad_(True)
    p = {k: leaf(k) for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")}
    if support == "dense":
        Gs = leaf("Gs")
        vals = None
    else:
        sp = t["Gs"].float().to_sparse_csr()
        vals = sp.values().to(DEV).requires_grad_(support == "learnable")
        Gs = S.CsrSupport(sp.crow_indices().int().to(DEV), sp.col_indices().int().to(DEV), vals, N)

    def step():
        _lib.set_concurrency(concurrency)
        for x in list(p.values()) + [Gs if support == "dense" else vals]:
            x.grad = None
        Hn = S.stc_cell_forward(Gs, p["Gc"], p["Xt"], p["H"], p["Wg"], p["bg"], p["Wc"], p["bc"], Ks, Kc)
        Hn.backward(t["dHn"].float().to(DEV))
        out = {"Hn": Hn, **{"d" + k: x.grad for k, x in p.items()}}
        out["dGs"] = Gs.grad if support == "dense" else vals.grad
        return out

    return t, cfg, step


def check_oracle(t, cfg, got, support):
    _, g = oracle_cell_with_grads(t, cfg)
    names = dict(dXt="dXt", dH="dH", dGc="dGc", dbg="dbg", dbc="dbc", dWg="dWg", dWc="dWc")
    for k, name in names.items():
        O.assert_close(got[k].cpu(), g[name], name, atol_scale=1e-5 if name in ("dWg", "dWc") else O.ATOL_SCALE)
    if support == "dense":
        O.assert_close(got["dGs"].cpu(), g["dGs"], "dGs")
    elif support == "learnable":
        sp = t["Gs"].float().to_sparse_csr()
        rows = torch.repeat_interleave(torch.arange(cfg["N"]), sp.crow_indices().diff())
        O.assert_close(got["dGs"].cpu(), g["dGs"][rows, sp.col_indices()], "dvals")


CELL_CASES = [
    # (B, N, C, Din, h, Ks, Kc), support, concurrency
    ((1024, 100, 5, 1, 16, 2, 2), "dense", -1),     # SF shape, lanes inactive (tc conv kernels, tc_outer slots)
    ((32, 100, 5, 16, 16, 2, 2), "dense", -1),      # small batch, lanes active
    ((64, 100, 5, 1, 16, 2, 2), "dense", 0),        # Din = 1, one stream
    ((4, 200, 4, 8, 16, 2, 2), "dense", -1),        # dense N = 200: block-wise tc_outer
    ((16, 60, 4, 64, 64, 2, 2), "dense", -1),       # wide state: the big dx / dW kernels
    ((8, 150, 5, 4, 16, 2, 2), "constant", 0),
    ((8, 150, 5, 4, 16, 2, 2), "constant", 1),
    ((8, 150, 5, 4, 16, 2, 2), "learnable", 0),
    ((8, 150, 5, 4, 16, 2, 2), "learnable", 1),     # both adjoint chains add into the edge gradient
    ((4, 20, 3, 2, 6, 2, 2), "dense", -1),          # h % 8 != 0: the general FFMA dx and dW kernels
    ((16, 20, 5, 1, 16, 3, 2), "dense", -1),        # Ks * (h + 8) > 64: tensor-core dx, general dW
    ((16, 20, 5, 1, 16, 2, 3), "dense", 0),         # Kc = 3: Kc * 2h > 64, general dW
    ((8, 150, 5, 4, 16, 3, 2), "learnable", 1),     # Ks = 3 with a learnable CSR support
]


@pytest.mark.parametrize("shape,support,conc", CELL_CASES)
def test_cell_is_bitwise_repeatable(deterministic, shape, support, conc):
    t, cfg, step = cell_case(shape, support, seed=sum(shape), concurrency=conc)
    got = repeat3(step)
    check_oracle(t, cfg, got, support)


def test_reduce_kernel_runs_only_in_deterministic_mode():
    _, _, step = cell_case((256, 100, 5, 1, 16, 2, 2))
    step()
    was = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        assert "det_reduce" not in kinds_of(step)
        torch.use_deterministic_algorithms(True)
        step()
        assert "det_reduce" in kinds_of(step)
    finally:
        torch.use_deterministic_algorithms(was)
        _lib.sync_deterministic()
        _lib.set_concurrency(-1)


def test_nan_prefilled_buffers_give_the_same_bits(deterministic):
    """The library never reads a float of `saved` / `scratch` it did not write: the deterministic results are bitwise the
    same whether torch fills fresh buffers with NaN or not."""
    import torch.utils.deterministic as D
    # SF (tc conv kernels, tc_outer slots for the H side, the FFMA support_outer slots for the 5-wide Xt side), the
    # wide-state kernels, block-wise tc_outer (N = 200), the general FFMA conv kernels, constant and learnable CSR
    for shape, support in (((512, 100, 5, 1, 16, 2, 2), "dense"), ((16, 60, 4, 64, 64, 2, 2), "dense"),
                           ((4, 200, 4, 8, 16, 2, 2), "dense"), ((4, 20, 3, 2, 6, 2, 2), "dense"),
                           ((16, 20, 5, 1, 16, 3, 2), "dense"), ((8, 150, 5, 4, 16, 2, 2), "constant"),
                           ((8, 150, 5, 4, 16, 2, 2), "learnable")):
        _, _, step = cell_case(shape, support, seed=1)
        fill = D.fill_uninitialized_memory
        try:
            D.fill_uninitialized_memory = True
            a = {k: v.detach().clone() for k, v in step().items() if v is not None}
            D.fill_uninitialized_memory = False
            b = {k: v.detach().clone() for k, v in step().items() if v is not None}
        finally:
            D.fill_uninitialized_memory = fill
        for k in a:
            assert torch.equal(a[k], b[k]), f"{shape} {support}: {k} depends on the NaN fill"
            assert torch.isfinite(a[k]).all(), k


@pytest.mark.parametrize("kind", ["dense", "csr_learned"])
def test_stack_with_shared_and_hoisted_terms(deterministic, kind):
    """RecurrentStack with shared terms (and, dense, the hoisted layer-0 product through stc_support_outer_ws): bitwise
    repeatable, and every gradient within the stack floor of the unshared cell-by-cell roll-out."""
    from tests.test_shared_terms_gpu import close, make_case, reference_rollout
    stack, Gs, Gc, X, dOut, leaves = make_case(kind, T=4, horizon=2, B=64)

    def step():
        for q in leaves:
            q.grad = None
        out = stack(Gs, Gc, X)
        out.backward(dOut)
        return {"out": out, **{f"g{i}": q.grad for i, q in enumerate(leaves)}}

    got = repeat3(step)
    for q in leaves:
        q.grad = None
    ref = reference_rollout(stack, Gs, Gc, X)
    ref.backward(dOut)
    close(got["out"], ref, "out")
    for i, q in enumerate(leaves):
        close(got[f"g{i}"], q.grad, f"grad {i}")


def test_graphed_step_replayed_three_times(deterministic):
    """GraphedStep captured in deterministic mode (the scratch slots and the NaN-filled buffers are allocated inside the
    capture) replays bitwise three times, and equals the eager deterministic step within the stack floor."""
    from tests.test_shared_terms_gpu import close, make_case
    stack, Gs, Gc, X0, dOut, leaves = make_case("dense", T=4, horizon=2, seed=5, B=32)
    X1 = (torch.rand(X0.shape, generator=torch.Generator().manual_seed(9)) < 0.3).float().to(DEV)
    loss_fn = lambda X: (stack(Gs, Gc, X) * dOut).sum()
    gs = S.GraphedStep(loss_fn, [X0], leaves)

    def step():
        loss = gs.replay(X1)
        return {"loss": loss, **{f"g{i}": q.grad for i, q in enumerate(leaves)}}

    got = repeat3(step)
    for q in leaves:
        q.grad = None
    loss_e = loss_fn(X1)
    loss_e.backward()
    assert abs(float(got["loss"]) - float(loss_e)) <= 1e-5 * abs(float(loss_e))
    for i, q in enumerate(leaves):
        close(got[f"g{i}"], q.grad, f"graphed grad {i}")


def test_partitioned_learnable_support_world_1(deterministic):
    """The halo path at world 1: its stages, row-list edge-gradient hops and torch ops (index_add_, integer cumsum,
    stable sort, bincount) all run under the switch and repeat bitwise."""
    import torch.distributed as dist
    if not dist.is_initialized():
        import tempfile
        f = tempfile.NamedTemporaryFile(delete=False)
        dist.init_process_group("gloo", init_method=f"file://{f.name}", rank=0, world_size=1)
    B, N, C, Din, h, Ks, Kc = 4, 120, 4, 4, 16, 2, 2
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=5, sparse_frac=0.9)
    sp = t["Gs"].float().to_sparse_csr()
    vals = torch.nn.Parameter(sp.values().to(DEV))
    ps = S.halo.PartitionedSupport(sp.crow_indices(), sp.col_indices(), vals, N, 0, 1)
    leaf = lambda k: t[k].float().to(DEV).requires_grad_(True)
    p = {k: leaf(k) for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")}

    def step():
        for x in list(p.values()) + [vals]:
            x.grad = None
        Hn = S.halo.partitioned_cell_forward(ps, p["Gc"], p["Xt"], p["H"], p["Wg"], p["bg"], p["Wc"], p["bc"], Ks, Kc)
        Hn.backward(t["dHn"].float().to(DEV))
        return {"Hn": Hn, "dvals": vals.grad, **{"d" + k: x.grad for k, x in p.items()}}

    got = repeat3(step)
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, activation=None)
    check_oracle(t, cfg, {**got, "dGs": got["dvals"]}, "learnable")


# ---- two ranks over gloo on one GPU: the interior / boundary row-list hops and the all-gathers run ----------------------
def _two_rank_worker(rank, world, port, q):
    import os
    import traceback
    import torch.distributed as dist
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        torch.use_deterministic_algorithms(True)
        from tests.learned_csr_oracle import stc_cell_edge_grad
        from tests.test_halo_learned_gpu import ARGS, learnable_partition
        from tests.test_learned_csr_gpu import dense_of, pattern
        B, N, C, Din, h, Ks, Kc = 2, 101, 5, 16, 16, 2, 2
        rowptr, col, vals = pattern(N, 6, seed=33, empty_every=9)
        t = random_case(B, N, C, Din, h, Ks, Kc, seed=33)
        t["Gs"] = dense_of(rowptr, col, vals, N)
        Hn_o, g_o = oracle_cell_with_grads(t, dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc))
        dv_o = stc_cell_edge_grad(torch.sparse_csr_tensor(rowptr.long(), col.long(), vals.double(), size=(N, N)),
                                  *(t[k] for k in ARGS), Ks, Kc, t["dHn"])
        ps, v = learnable_partition(rowptr, col, vals, N, rank, world, DEV)
        assert ps.fwd.nhalo > 0
        loc = lambda k: ps.local_slice(t[k]) if k in ("Xt", "H", "dHn") else t[k]
        p = {k: loc(k).float().to(DEV).requires_grad_(True) for k in ARGS}

        def step():
            for x in list(p.values()) + [v]:
                x.grad = None
            out = S.halo.partitioned_cell_forward(ps, *(p[k] for k in ARGS), Ks, Kc)
            out.backward(loc("dHn").float().to(DEV))
            return {"Hn": out, "dvals": v.grad, **{"d" + k: x.grad for k, x in p.items()}}

        got = repeat3(step)
        O.assert_close(got["Hn"].cpu(), ps.local_slice(Hn_o), "H'")
        O.assert_close(got["dvals"].cpu(), dv_o, "dvals")
        for k, name in (("Xt", "dXt"), ("H", "dH")):
            O.assert_close(got["d" + k].cpu(), ps.local_slice(g_o[name]), name)
        for k, name in (("Wg", "dWg"), ("Wc", "dWc"), ("bg", "dbg"), ("bc", "dbc"), ("Gc", "dGc")):
            O.assert_close(got["d" + k].cpu(), g_o[name], name)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, None))
    except Exception:  # pragma: no cover - reported by the parent
        q.put((rank, traceback.format_exc()))


def test_partitioned_learnable_support_two_ranks_gloo():
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    try:
        results = [q.get(timeout=600) for _ in procs]
    finally:
        for pr in procs:
            pr.join(timeout=60)
            if pr.is_alive():
                pr.terminate()
                pr.join()
    for rank, err in results:
        assert err is None, f"rank {rank}:\n{err}"


# ---- the sparse graph generator: cuBLAS runs inside it, so CUBLAS_WORKSPACE_CONFIG is set before CUDA starts ------------
def _generator_child():
    from tests import sparse_mgp_oracle as SO
    from tests.test_sparse_mgp_gpu import csr
    torch.use_deterministic_algorithms(True)
    N, C, Ks, Kc, h, layers, horizon, B, T, hg = 48, 3, 2, 2, 8, 2, 2, 2, 3, 4
    g = torch.Generator().manual_seed(41)
    X = torch.randn(B, T, N, C, generator=g)
    Gc = (torch.rand(C, C, generator=g) / C).to(DEV)
    dOut = torch.randn(B, horizon, N, C, h, generator=g).to(DEV)
    torch.manual_seed(41)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    stack = S.RecurrentStack(N, C, Ks, Kc, 1, h, layers, horizon).to(DEV)
    rowptr, col = SO.random_pattern(N, 6, seed=2, empty_every=9)
    pat = csr(rowptr, col)
    leaves = list(gen.parameters()) + list(stack.parameters())
    for mode in ("pattern", "k"):
        def step():
            for x in leaves:
                x.grad = None
            sup = gen(X.to(DEV), pat) if mode == "pattern" else gen(X.to(DEV), k=8)
            out = stack(sup, Gc, X.to(DEV)[..., None])
            out.backward(dOut)
            return {"out": out, "vals": sup.vals, **{f"g{i}": x.grad for i, x in enumerate(leaves)}}
        got = repeat3(step)
        if mode == "pattern":   # the generated values against the fp64 generator on the same pattern
            Wu64 = gen.params_S["Wu"].detach().double().cpu()
            Wv64 = gen.params_S["Wv"].detach().double().cpu()
            P64 = SO.sparse_generator(X.double(), Wu64, Wv64, gen.alpha, rowptr, col)
            O.assert_close(got["vals"].cpu(), P64, "generated values")
        print(f"generator {mode}: bitwise over three runs", flush=True)


def test_sparse_graph_generator_in_child():
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    code = (f"import sys; sys.path.insert(0, {root!r}); from tests.test_deterministic_gpu import _generator_child; "
            "_generator_child()")
    res = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=900)
    print(res.stdout[-3000:])
    assert res.returncode == 0, f"child exited with {res.returncode}\n{res.stdout[-3000:]}\n{res.stderr[-5000:]}"
