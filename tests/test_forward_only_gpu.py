"""The forward-only cell calls (stc_cell_fwd_only*, chosen when no gradient can be asked for) against the training
forward: H' and every roll-out built from it must be BITWISE the grad-enabled result -- the arithmetic is the same, only
the stores the backward needs (r, c, the P_1 partials) are dropped -- the same forward convolution kernels run, and the
workspace is the smaller one."""
import os
import socket
import traceback

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import stc_gnn_b200 as S
from stc_gnn_b200 import _lib, cell
from stc_gnn_b200.synth import sf_supports
from tests.helpers import random_case
from tests.test_conv_variants_gpu import CASES, batch_of, cell_step, device_leaves, make_inputs, record_conv_kernels

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def fwd_only_calls(fn):
    """fn()'s result and whether a forward-only workspace size was looked up while it ran."""
    cell._SIZES.clear()
    out = fn()
    return out, any(k[0] == "fwd_only" for k in cell._SIZES)


def conv_kernels(fn, calls=3):
    """fn()'s last result and the convolution kernels the profiler saw over `calls` calls: a session that holds only one
    short forward has been seen to lose the records of its first kernels, so the set is taken over repeated calls."""
    return record_conv_kernels(lambda: [fn() for _ in range(calls)][-1])


# ---- 1. every convolution kernel variant ----------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_every_variant_is_bitwise(name):
    spec = CASES[name]
    t, _ = make_inputs(spec, batch_of(spec), seed=len(name) + 3)
    v = device_leaves(t, spec)
    want, k_train = conv_kernels(lambda: cell_step(v, spec))
    assert want.requires_grad
    with torch.no_grad():
        (got, k_fwd), used = fwd_only_calls(lambda: conv_kernels(lambda: cell_step(v, spec)))
    assert used and not got.requires_grad
    assert k_fwd == k_train and k_fwd, (name, k_fwd, k_train)
    assert torch.equal(got, want.detach()), f"{name}: {(got - want).abs().max().item():.3e}"


# ---- 2. dense N = 200, constant and learnable CSR, timing kinds --------------------------------------------------------
def _leaves(B, N, C, Din, h, Ks, Kc, seed, sparse=None):
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=seed, sparse_frac=sparse)
    return t, {k: t[k].float().to(DEV).requires_grad_(True) for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")}


def _both(Gs, v, Ks, Kc):
    args = lambda: (Gs, v["Gc"], v["Xt"], v["H"], v["Wg"], v["bg"], v["Wc"], v["bc"], Ks, Kc)
    want = S.stc_cell_forward(*args())
    with torch.no_grad():
        got, used = fwd_only_calls(lambda: S.stc_cell_forward(*args()))
    assert used
    return want.detach(), got


def test_dense_n200_with_the_same_timing_kinds():
    B, N, C, Din, h, Ks, Kc = 4, 200, 5, 16, 16, 3, 2
    t, v = _leaves(B, N, C, Din, h, Ks, Kc, seed=1)
    Gs = t["Gs"].float().to(DEV).requires_grad_(True)
    _both(Gs, v, Ks, Kc)   # warm
    kinds = []
    for grad in (True, False):
        _lib.timing_enable(True)
        _lib.timing_collect()
        with torch.set_grad_enabled(grad):
            out = S.stc_cell_forward(Gs, v["Gc"], v["Xt"], v["H"], v["Wg"], v["bg"], v["Wc"], v["bc"], Ks, Kc)
        torch.cuda.synchronize()
        _lib.timing_enable(False)
        kinds.append((out.detach(), _lib.timing_collect()))
    (want, k_train), (got, k_fwd) = kinds
    assert torch.equal(got, want)
    assert {k: c for k, (_, c, _) in k_fwd.items()} == {k: c for k, (_, c, _) in k_train.items()}
    # the algorithmic bytes of the forward convolutions drop by exactly r and c (one float each per row and channel)
    conv = next(k for k in k_train if "conv_fwd" in k)
    assert k_train[conv][2] - k_fwd[conv][2] == 4 * (B * N * C) * 2 * h, (k_train[conv], k_fwd[conv])


@pytest.mark.parametrize("learnable", [False, True])
def test_csr_supports(learnable):
    B, N, C, Din, h, Ks, Kc = 3, 64, 4, 3, 8, 3, 2
    t, v = _leaves(B, N, C, Din, h, Ks, Kc, seed=2, sparse=0.85)
    s = t["Gs"].float().to(DEV).to_sparse_csr()
    vals = s.values().clone().requires_grad_(learnable)
    Gs = S.CsrSupport(s.crow_indices(), s.col_indices(), vals, N)
    want, got = _both(Gs, v, Ks, Kc)
    assert torch.equal(got, want)


# ---- 3. roll-outs ----------------------------------------------------------------------------------------------------
ROLLOUTS = {"sf_hoisted": dict(kind="dense"), "dense_ks3": dict(kind="dense", Ks=3, T=4, horizon=2),
            "csr": dict(kind="csr_learned", T=4, horizon=2), "layers3": dict(kind="dense", layers=3, T=3, horizon=2),
            "horizon0": dict(kind="dense", T=5, horizon=0)}


@pytest.mark.parametrize("name", list(ROLLOUTS))
def test_recurrent_stack_rollouts(name):
    from tests.test_shared_terms_gpu import make_case
    stack, Gs, Gc, X, _, _ = make_case(**ROLLOUTS[name])
    want = stack(Gs, Gc, X)
    assert want.requires_grad
    with torch.no_grad():
        got, used = fwd_only_calls(lambda: stack(Gs, Gc, X))
    assert used
    assert torch.equal(got, want.detach())


def test_generator_and_stack_under_no_grad():
    from tests import sparse_mgp_oracle as SO
    B, T, N, C, hg, h = 2, 4, 64, 3, 4, 8
    g = torch.Generator().manual_seed(6)
    X = torch.randn(B, T, N, C, generator=g).to(DEV)
    torch.manual_seed(6)
    gen = S.SparseGraphGenerator(C, hg).to(DEV)
    stack = S.RecurrentStack(N, C, 3, 2, 1, h, 2, 2).to(DEV)
    rowptr, col = SO.random_pattern(N, 6, seed=6)
    pat = S.CsrSupport(rowptr.to(DEV), col.to(DEV), torch.ones(col.numel(), device=DEV), N)
    Gc = (torch.rand(C, C, generator=g) / C).to(DEV)
    run = lambda: stack(gen(X, pat), Gc, X.unsqueeze(-1))
    want = run()
    with torch.no_grad():
        got, used = fwd_only_calls(run)
    assert used
    assert torch.equal(got, want.detach())


# ---- 4. the row partition ----------------------------------------------------------------------------------------------
def _partitioned_bitwise(rank, world, dev, seed):
    B, N, C, Din, h, Ks, Kc = 2, 96, 5, 16, 16, 3, 2
    t, _ = _leaves(B, N, C, Din, h, Ks, Kc, seed=seed, sparse=0.85)
    ps = S.halo.PartitionedSupport.from_dense(t["Gs"], rank, world)
    f = lambda k: (ps.local_slice(t[k]) if k in ("Xt", "H") else t[k]).float().to(dev).requires_grad_(True)
    v = {k: f(k) for k in ("Gc", "Xt", "H", "Wg", "bg", "Wc", "bc")}
    run = lambda: S.halo.partitioned_cell_forward(ps, v["Gc"], v["Xt"], v["H"], v["Wg"], v["bg"], v["Wc"], v["bc"], Ks, Kc)
    want = run()
    assert want.requires_grad
    with torch.no_grad():
        got = run()
    assert torch.equal(got, want.detach()), f"rank {rank}/{world}"
    return ps


def test_partitioned_cell_world_1():
    _partitioned_bitwise(0, 1, DEV, seed=4)


def _two_rank_worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        ps = _partitioned_bitwise(rank, world, torch.device("cuda", 0), seed=5)
        assert ps.fwd.nhalo > 0
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, None))
    except Exception:  # pragma: no cover - reported by the parent
        q.put((rank, traceback.format_exc()))


def test_partitioned_cell_two_ranks_gloo_one_gpu():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, q)) for r in range(2)]
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


# ---- 5. memory, the deterministic mode's NaN fill, the switch, a short workspace ---------------------------------------
def _sf_cell(B):
    torch.manual_seed(0)
    c = S.STC_Cell(100, 5, 2, 2, 16, 16).to(DEV)
    Gs, Gc = (x.to(DEV) for x in sf_supports(seed=0))
    g = torch.Generator().manual_seed(1)
    Xt = torch.randn(B, 100, 5, 16, generator=g).to(DEV)
    H = torch.randn(B, 100, 5, 16, generator=g).to(DEV)
    return c, Gs, Gc, Xt, H


def test_peak_memory_of_a_no_grad_sf_call():
    B = 4096
    c, Gs, Gc, Xt, H = _sf_cell(B)
    with torch.no_grad():
        c(Gs, Gc, Xt, H)   # warm
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = c(Gs, Gc, Xt, H)
        torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    d = _lib.StcDims(B, 100, 5, 16, 16, 2, 2, 0, 1)
    lib = _lib.load()
    ws, saved = lib.stc_cell_fwd_only_bytes(d), lib.stc_cell_saved_bytes(d)
    slack = 2 * (2 << 20)   # the caching allocator rounds each large block up to a multiple of 2 MiB
    assert grown <= ws + out.numel() * 4 + slack, (grown, ws, out.numel() * 4)
    assert grown < saved, (grown, saved)


def test_nan_filled_workspace_gives_the_same_bits():
    """torch.use_deterministic_algorithms(True) NaN-fills every fresh buffer: the forward reads nothing it did not write."""
    c, Gs, Gc, Xt, H = _sf_cell(64)
    want = c(Gs, Gc, Xt, H).detach()
    was, fill = torch.are_deterministic_algorithms_enabled(), torch.utils.deterministic.fill_uninitialized_memory
    try:
        torch.use_deterministic_algorithms(True)
        torch.utils.deterministic.fill_uninitialized_memory = True
        with torch.no_grad():
            got, used = fwd_only_calls(lambda: c(Gs, Gc, Xt, H))
    finally:
        torch.use_deterministic_algorithms(was)
        torch.utils.deterministic.fill_uninitialized_memory = fill
        _lib.sync_deterministic()
    assert used and not torch.isnan(got).any()
    assert torch.equal(got, want)


def test_switch_off_keeps_the_training_forward(monkeypatch):
    c, Gs, Gc, Xt, H = _sf_cell(16)
    with torch.no_grad():
        a = c(Gs, Gc, Xt, H)
        monkeypatch.setattr(cell, "FORWARD_ONLY", False)
        b, used = fwd_only_calls(lambda: c(Gs, Gc, Xt, H))
    assert not used
    assert torch.equal(a, b)


def test_too_small_workspace_is_refused():
    B, N, C, Din, h, Ks, Kc = 2, 100, 5, 16, 16, 2, 2
    t, v = _leaves(B, N, C, Din, h, Ks, Kc, seed=3)
    lib = _lib.load()
    d = _lib.StcDims(B, N, C, Din, h, Ks, Kc, 0, 1)
    need = lib.stc_cell_fwd_only_bytes(d)
    ws = torch.empty(need // 4, device=DEV)
    Gs = t["Gs"].float().to(DEV)
    out = torch.empty(B, N, C, h, device=DEV)
    p = lambda k: v[k].data_ptr()
    args = (d, S.support.dense_struct(Gs), p("Gc"), p("Xt"), N * C * Din, p("H"), p("Wg"), p("bg"), p("Wc"), p("bc"),
            out.data_ptr(), ws.data_ptr())
    status = lib.stc_cell_fwd_only(*args, need - 4, None, None, None)
    with pytest.raises(RuntimeError, match="STC_ERR_WORKSPACE"):
        _lib.check(status, "stc_cell_fwd_only")
    status = lib.stc_cell_fwd_only_stage(d, _lib.STAGE_GATES, p("Gc"), p("Xt"), N * C * Din, p("H"), p("Wg"), p("bg"),
                                         p("Wc"), p("bc"), out.data_ptr(), ws.data_ptr(), need - 4, None)
    assert status == -3 and b"STC_ERR_WORKSPACE" in lib.stc_last_error()


# ---- 6. the full reference model with the cell installed ---------------------------------------------------------------
def test_installed_full_model_predictions_under_no_grad():
    from tests.helpers import find_reference, import_reference
    if find_reference() is None:
        pytest.skip("the unmodified reference is not on this box (tools/stage_reference.sh stages it under baseline/_ref)")
    from tests.test_dropin_gpu import _first_train_batch
    from stc_gnn_b200.install import install, uninstall
    ref, ref_dir = import_reference()
    X, _, As, Ac = _first_train_batch(ref_dir)
    install(ref)
    try:
        torch.manual_seed(0)
        model = ref.STCGNN(100, 5, 2, 2, 1, 16, 2, 3).to(DEV)
    finally:
        uninstall(ref)
    want = model(X_seq=X, As=As, Ac=Ac)
    assert want.requires_grad
    with torch.no_grad():
        got, used = fwd_only_calls(lambda: model(X_seq=X, As=As, Ac=Ac))
    assert used
    assert torch.equal(got, want.detach())
