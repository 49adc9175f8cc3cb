"""Every convolution kernel variant against the fp64 oracle, at sizes where each persistent CTA runs several tiles.

One cell step launches a forward, an input adjoint (dx) and a weight gradient (dW) convolution per gate pass, and the
host picks each from a ladder of kernels by shape, alignment and switches.  The kernels that actually ran are read back
from the CUDA profiler -- the dispatch is not restated here -- and each case declares the exact set it must launch, so a
case that silently moves to another variant fails instead of passing on a path nobody meant to test.

Tolerances: element-wise tensors keep the per-cell 1e-4 |ref| + 1e-5 mean|ref|.  Reduced tensors (dW, db, dGs / edge
values, dGc) of a case with more than 30 K rows may use 3e-5 mean|ref| (the config 3 precedent in test_cell_gpu.py);
such a case prints the deviation of an fp32 evaluation of the reference's operator sequence from fp64 beside it."""
import os
import re
import subprocess
import sys

import pytest
import torch

from oracle import stc_oracle as O
from tests.helpers import oracle_cell_with_grads, random_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ---- the convolution kernel instantiations of libstc_b200.so (tests/test_conv_variants_cpu.py checks this list) ----
F_AT1, F_AT2 = "tc_conv_fwd_at_kernel<1>", "tc_conv_fwd_at_kernel<2>"
F_TC0, F_TC1, F_TC2 = "tc_conv_fwd_kernel<0>", "tc_conv_fwd_kernel<1>", "tc_conv_fwd_kernel<2>"
F_BIG = "tc_conv_fwd_big_kernel"
F_FF1, F_FF2, F_FF4 = "conv_fwd_kernel<1>", "conv_fwd_kernel<2>", "conv_fwd_kernel<4>"
DX_AT, DX_FAST, DX_GEN = "tc_conv_bwd_dx_kernel<true, true>", "tc_conv_bwd_dx_kernel<true, false>", \
    "tc_conv_bwd_dx_kernel<false, false>"
DX_BIG = "tc_conv_bwd_dx_big_kernel"
DX_FF1, DX_FF2, DX_FF4 = "conv_bwd_dx_kernel<1>", "conv_bwd_dx_kernel<2>", "conv_bwd_dx_kernel<4>"
DWP1, DWP2, DWP4 = "tc_conv_bwd_dw_pipe_kernel<1>", "tc_conv_bwd_dw_pipe_kernel<2>", "tc_conv_bwd_dw_pipe_kernel<4>"
DW1, DW2, DW4 = "tc_conv_bwd_dw_kernel<1>", "tc_conv_bwd_dw_kernel<2>", "tc_conv_bwd_dw_kernel<4>"
DW_BIG = "tc_conv_bwd_dw_big_kernel"
DW_FF1, DW_FF2, DW_FF4 = "conv_bwd_dw_kernel<1>", "conv_bwd_dw_kernel<2>", "conv_bwd_dw_kernel<4>"
VARIANTS = [F_AT1, F_AT2, F_TC0, F_TC1, F_TC2, F_BIG, F_FF1, F_FF2, F_FF4, DX_AT, DX_FAST, DX_GEN, DX_BIG, DX_FF1,
            DX_FF2, DX_FF4, DWP1, DWP2, DWP4, DW1, DW2, DW4, DW_BIG, DW_FF1, DW_FF2, DW_FF4]
# instantiations no shape reaches, with the launch condition that rules each out (none at present)
EXCLUDED = {}

_CONV_NAME = re.compile(r"(?:void\s+)?(?:stc::)?(\w*conv\w*_kernel(?:<[^()]*>)?)\s*\(")


def conv_kernel_name(demangled):
    """'void stc::tc_conv_bwd_dx_kernel<true, false>(stc::ConvArgs, stc::TcDxPlan)' -> 'tc_conv_bwd_dx_kernel<true, false>'
    (None for kernels that are not convolutions)."""
    m = _CONV_NAME.match(demangled.strip())
    return m.group(1) if m else None


# ---- multi-tile sizing -------------------------------------------------------------------------------------------------
DW_TR = 64          # rows of one tensor-core dW tile
MAX_CTAS_PER_SM = 2  # the largest persistent grid any convolution kernel launches is 2 CTAs per SM


def multi_tile_batch(N, C, sms, min_tiles_per_cta=3):
    """Smallest batch at which every persistent convolution kernel runs >= 3 tiles per CTA even on its largest grid
    (2 CTAs per SM): the forward / dx tiles hold 128 // C whole nodes, the dW tiles 64 rows of B*N*C.  The batch is
    then raised until the last wave is partial (tile count not a multiple of the grid) and, where N allows it, the last
    node tile is ragged (B*N not a multiple of 128 // C).  Returns (B, tiles per CTA of the node tiles, of the dW tiles)."""
    grid, npt = MAX_CTAS_PER_SM * sms, 128 // C
    B = 1
    while (B * N + npt - 1) // npt < min_tiles_per_cta * grid or (B * N * C + DW_TR - 1) // DW_TR < min_tiles_per_cta * grid:
        B += 1
    ragged_possible = any((b * N) % npt for b in range(1, npt + 1))
    for b in range(B, B + 4 * npt * grid):
        tiles = (b * N + npt - 1) // npt
        if tiles % grid and (not ragged_possible or (b * N) % npt) and ((b * N * C + DW_TR - 1) // DW_TR) % grid:
            B = b
            break
    return B, ((B * N + npt - 1) // npt) / grid, ((B * N * C + DW_TR - 1) // DW_TR) / grid


# ---- the case table -----------------------------------------------------------------------------------------------------
def case(N, C, Din, h, Ks, Kc, kernels, B=None, bias=True, act=None, gs="dense", strided=False):
    """B = None: sized by multi_tile_batch on this device.  gs: "dense" or "csr" (learnable edge values).  strided: Xt
    is the [:, 1] view of a [B, 3, N, C, Din] sequence -- the layout RecurrentStack passes; with N*C*Din odd its batch
    stride is not a multiple of 4 and its base is not 16-byte aligned."""
    return dict(N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, B=B, bias=bias, act=act, gs=gs, strided=strided,
                kernels=frozenset(kernels))


SF_AT = {F_AT1, F_AT2, DX_AT}
CASES = {
    # ---- multi-tile: every instantiation with >= 3 tiles per CTA, partial last wave, ragged last tile ----------------
    "mt_sf_din16": case(100, 5, 16, 16, 2, 2, SF_AT | {DWP2, DWP4}),                       # the benchmark's SF shape
    "mt_sf_din1_csr_strided_relu": case(101, 5, 1, 16, 2, 2, SF_AT | {DW2, DW4}, act="relu", gs="csr", strided=True),
    "mt_sf_din1_n99": case(99, 5, 1, 16, 2, 2, SF_AT | {DW2, DW4}),                        # N*C*Din % 4 != 0: no dW pipe
    "mt_c7_nobias": case(100, 7, 16, 16, 2, 2, SF_AT | {DWP2, DWP4}, bias=False),          # 126 of 128 tile rows
    "mt_kc1": case(99, 5, 1, 16, 2, 1, {F_TC0, DX_FAST, DW1, DW2}),
    "mt_kc1_pipe": case(101, 5, 4, 16, 2, 1, {F_TC0, DX_FAST, DWP1, DWP2}),      # C*Din = 20: width % 8 == 4 for dGs
    "mt_kc3": case(100, 5, 4, 16, 2, 3, {F_TC0, DX_FAST, DWP4, DW_FF1}),
    "mt_ks3_nobias": case(100, 5, 16, 16, 3, 2, {F_TC1, F_TC2, DX_GEN, DW_FF1}, bias=False),
    # (ReLU stays off at this size on a dense support: among ~10^7 pre-activations a few lie within fp32 rounding of
    #  zero, so the mask flips and the dense hop spreads the flip over whole rows -- the fp32 evaluation of the
    #  reference itself then deviates 1e-3 x mean|ref| in dWg from fp64.  ReLU is checked on every tier at small B.)
    "mt_big": case(40, 8, 1, 64, 2, 2, {F_BIG, DX_BIG, DW_BIG}),
    "mt_h80_two_tiers": case(97, 5, 16, 80, 2, 2, {F_FF4, F_BIG, DX_FF1, DX_BIG, DW_FF2, DW_BIG}),
    # C*h = 84: the H-side dGs product has width % 8 == 4 with more samples than CTAs (stale-column read, fixed)
    "mt_ffma_din3_strided": case(101, 7, 3, 12, 2, 2, {F_FF1, F_FF2, DX_FF1, DW_FF1}, strided=True),
    "mt_ffma_wide_l": case(31, 5, 89, 40, 2, 2, {F_FF1, F_FF2, DX_FF2, DW_FF2, DW_FF4}),
    "mt_ffma_dx4": case(29, 64, 121, 8, 2, 2, {F_FF1, DX_FF4, DW_FF1}),                      # one 64-row node per dx tile
    # ---- boundary pairs, one case on each side of a cut (small batches) -----------------------------------------------
    # tensor-memory columns of dx, (KA + 1) * ceil16(Ks * KBL) <= 512: Ks = 6 is the last eligible value at h = 16,
    # Din = 1; at Ks = 7 the gates pass leaves the tensor cores while the candidate pass (half the columns) stays
    "ks6_tmem_last": case(30, 5, 1, 16, 6, 2, {F_TC0, DX_GEN, DW_FF1}, B=3),
    "ks7_tmem_next": case(30, 5, 1, 16, 7, 2, {F_TC0, DX_GEN, F_FF2, DX_FF1, DW_FF1}, B=3),
    # KB = 1 -> 2: Din 16 -> 17 moves the forward from the A-in-TMEM kernel to the generic one
    "din17_kb2": case(33, 5, 17, 16, 2, 2, {F_TC0, DX_GEN, DW_FF1}, B=3),
    # KBLp = ceil16(h + ceil8(Din)) 128 -> 144: the wide-state dx / dW of the candidate pass fall back to FFMA
    "h112_kblp128": case(20, 8, 16, 112, 2, 2, {F_FF2, F_BIG, DX_FF1, DX_BIG, DW_FF2, DW_BIG}, B=2),
    "h112_kblp144_din17": case(20, 8, 17, 112, 2, 2, {F_FF2, F_BIG, DX_FF1, DX_FF2, DW_FF4}, B=2),
    # Hout 128 -> 160, the wide-state limit: h = 64 runs both passes wide, h = 80 the candidate only
    "h64_hout128": case(21, 5, 16, 64, 2, 2, {F_BIG, DX_BIG, DW_BIG}, B=3),
    "h80_hout160": case(21, 5, 16, 80, 2, 2, {F_FF4, F_BIG, DX_FF1, DX_BIG, DW_FF2, DW_BIG}, B=3),
    # hidden widths: h = 8 gates on the tensor cores / candidate on FFMA, h = 24 likewise, h = 32 gates wide / candidate
    # on the tensor cores, h = 48 wide in both passes
    "h8_split": case(33, 5, 4, 8, 2, 2, {F_TC1, DX_GEN, DWP2, F_FF1, DX_FF1, DW_FF1}, B=3),
    "h24_split": case(33, 5, 4, 24, 2, 2, {F_TC0, DX_GEN, F_FF2, DX_FF1, DW_FF1}, B=3),
    "h32_split": case(33, 5, 1, 32, 2, 2, {F_BIG, DX_BIG, DW_BIG, F_TC0, DX_GEN, DW_FF1}, B=3),
    "h48_big": case(21, 5, 20, 48, 2, 2, {F_BIG, DX_BIG, DW_BIG}, B=3),
    # categorical / spatial orders
    "kc4": case(33, 5, 16, 16, 2, 4, {F_TC0, DX_GEN, DX_FAST, DWP4, DW_FF1}, B=3),
    "ks1": case(33, 5, 16, 16, 1, 2, {F_TC1, F_TC2, DX_GEN, DWP2, DWP4}, B=3),
    "ks5_din1": case(33, 5, 1, 16, 5, 2, {F_TC0, DX_GEN, DW_FF1}, B=3),
    # category counts: 126 of 128 rows (C = 3), two nodes per tile (C = 64), the largest C of the SF-family kernels
    # (gates dx shared memory) and one more, the largest C of the wide-state kernels (gates forward shared memory)
    # and one more
    "c3": case(50, 3, 16, 16, 2, 2, SF_AT | {DWP2, DWP4}, B=3),
    "c64": case(9, 64, 16, 16, 2, 2, SF_AT | {DWP2, DWP4}, B=2),
    "c77_tc_max": case(5, 77, 16, 16, 2, 2, SF_AT | {DWP2, DWP4}, B=2),
    "c78_tc_next": case(5, 78, 16, 16, 2, 2, {F_AT1, DX_AT, DWP2, F_FF2, DX_FF1, DW_FF1}, B=2),
    "c70_big_max": case(4, 70, 16, 64, 2, 2, {F_BIG, DX_BIG, DW_BIG}, B=2),
    "c71_big_next": case(4, 71, 16, 64, 2, 2, {F_FF4, DX_FF2, DW_FF2, F_BIG, DX_BIG, DW_BIG}, B=2),
    # input layouts and epilogue options on each tier
    "tc_din3_strided_nobias": case(33, 5, 3, 16, 2, 2, SF_AT | {DW2, DW4}, B=3, bias=False, strided=True),
    "tc_din4_relu": case(33, 5, 4, 16, 2, 2, SF_AT | {DWP2, DWP4}, B=3, act="relu"),
    "big_din3_strided_nobias": case(33, 5, 3, 64, 2, 2, {F_BIG, DX_BIG, DW_BIG}, B=3, bias=False, strided=True),
    "big_din4_relu_nobias": case(21, 5, 4, 48, 2, 2, {F_BIG, DX_BIG, DW_BIG}, B=3, act="relu", bias=False),
    "ffma_din1_relu_nobias": case(33, 5, 1, 12, 2, 2, {F_FF1, F_FF2, DX_FF1, DW_FF1}, B=3, act="relu", bias=False),
    "ffma_din4_relu": case(33, 5, 4, 7, 2, 3, {F_FF1, DX_FF1, DW_FF1}, B=3, act="relu"),
}
MULTI_TILE = [k for k, v in CASES.items() if v["B"] is None]


def batch_of(spec, sms=None):
    if spec["B"] is not None:
        return spec["B"]
    return multi_tile_batch(spec["N"], spec["C"], sms or torch.cuda.get_device_properties(0).multi_processor_count)[0]


# ---- running one case ---------------------------------------------------------------------------------------------------
def make_inputs(spec, B, seed):
    N, C, Din, h, Ks, Kc = (spec[k] for k in ("N", "C", "Din", "h", "Ks", "Kc"))
    t = random_case(B, N, C, Din, h, Ks, Kc, seed=seed, use_bias=spec["bias"],
                    sparse_frac=0.85 if spec["gs"] == "csr" else None)
    cfg = dict(B=B, N=N, C=C, Din=Din, h=h, Ks=Ks, Kc=Kc, activation=spec["act"])
    return t, cfg


def device_leaves(t, spec):
    """fp32 CUDA leaves of a case (Xt as the strided view of a longer sequence when the case asks for it)."""
    leaf = lambda x: x.float().to(DEV).requires_grad_(True)
    v = {k: leaf(t[k]) for k in ("Gc", "H", "Wg", "Wc")}
    if spec["bias"]:
        v["bg"], v["bc"] = leaf(t["bg"]), leaf(t["bc"])
    if spec["strided"]:
        seq = torch.zeros(t["Xt"].shape[0], 3, *t["Xt"].shape[1:], device=DEV)
        seq[:, 1] = t["Xt"].float().to(DEV)
        v["_Xseq"] = seq.requires_grad_(True)
        v["Xt"] = seq[:, 1]
        assert v["Xt"].stride(0) % 4 != 0 and v["Xt"].data_ptr() % 16 != 0, "the view must be unaligned, odd-strided"
    else:
        v["Xt"] = leaf(t["Xt"])
    if spec["gs"] == "csr":
        Gd = t["Gs"].float().to(DEV)
        s = Gd.to_sparse_csr()
        v["vals"] = s.values().clone().requires_grad_(True)
        import stc_gnn_b200 as S
        v["Gs"] = S.CsrSupport(s.crow_indices(), s.col_indices(), v["vals"], Gd.shape[0])
        v["_csr"] = (s.crow_indices().cpu(), s.col_indices().cpu())
    else:
        v["Gs"] = leaf(t["Gs"])
    return v


def cell_step(v, spec, with_grad=True):
    import stc_gnn_b200 as S
    return S.stc_cell_forward(v["Gs"], v["Gc"], v["Xt"], v["H"], v["Wg"], v.get("bg"), v["Wc"], v.get("bc"),
                              spec["Ks"], spec["Kc"], spec["act"])


def record_conv_kernels(fn):
    """Run fn() once under the CUDA profiler; returns (fn's result, set of convolution kernel names that ran).  The step
    certainly launches kernels, so a trace without any device kernel is a broken recording, not an empty set."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    if not names:
        names = [e.name for e in prof.events()]
    conv = {n for n in (conv_kernel_name(x) for x in names) if n}
    if not any("_kernel" in x for x in names):
        pytest.fail(f"the profiler recorded no device kernel for a cell step that launches several (events: {names[:8]})")
    return out, conv


def run_case(spec, B, seed):
    """Forward + backward of one case under the profiler.  Returns (inputs, cfg, Hn, grads on the host, kernels)."""
    t, cfg = make_inputs(spec, B, seed)
    v = device_leaves(t, spec)
    dHn = t["dHn"].float().to(DEV)

    def step():
        Hn = cell_step(v, spec)
        Hn.backward(dHn)
        return Hn

    Hn, kernels = record_conv_kernels(step)
    g = dict(dH=v["H"].grad, dWg=v["Wg"].grad, dWc=v["Wc"].grad, dGc=v["Gc"].grad)
    if spec["strided"]:
        g["dXt"] = v["_Xseq"].grad[:, 1]
    else:
        g["dXt"] = v["Xt"].grad
    if spec["bias"]:
        g.update(dbg=v["bg"].grad, dbc=v["bc"].grad)
    if spec["gs"] == "csr":
        g["dvals"] = v["vals"].grad
    else:
        g["dGs"] = v["Gs"].grad
    return t, cfg, v, Hn.detach().cpu(), {k: x.detach().cpu() for k, x in g.items()}, kernels


def check_kernels(name, want, got):
    if got != want:
        pytest.fail(f"{name}: the convolution kernels that ran differ from the case table -- the table is stale or the "
                    f"dispatch moved.\n  ran but not declared: {sorted(got - want)}\n  declared but did not run: "
                    f"{sorted(want - got)}\n  ran: {sorted(got)}")


REDUCED = ("dWg", "dWc", "dbg", "dbc", "dGs", "dvals", "dGc")


def fp32_reference_floor(t, cfg):
    """Worst deviation (x mean|ref|) of an fp32 CPU evaluation of the reference's operator sequence from fp64, per
    reduced gradient: the arithmetic's own floor at this size."""
    def grads(dtype):
        names = ["Gs", "Gc", "Xt", "H", "Wg", "Wc"] + (["bg", "bc"] if t.get("bg") is not None else [])
        v = {k: t[k].to(dtype).clone().requires_grad_(True) for k in names}
        Hn = O.stc_cell_refshape(v["Gs"], v["Gc"], v["Xt"], v["H"], v["Wg"], v.get("bg"), v["Wc"], v.get("bc"),
                                 cfg["Ks"], cfg["Kc"], cfg.get("activation"))
        Hn.backward(t["dHn"].to(dtype))
        return {"d" + k: v[k].grad.double() for k in names if k not in ("Xt", "H") and v[k].grad is not None}
    lo, hi = grads(torch.float32), grads(torch.float64)
    return {k: (lo[k] - hi[k]).abs().max().item() / max(hi[k].abs().mean().item(), 1e-300) for k in hi}


def compare_with_oracle(name, t, cfg, v, Hn, g, spec):
    Hn_o, g_o = oracle_cell_with_grads(t, cfg)
    rows = cfg["B"] * cfg["N"] * cfg["C"]
    many = rows > 30000
    if spec["gs"] == "csr":
        crow, col = v["_csr"]
        row = torch.repeat_interleave(torch.arange(crow.numel() - 1), crow[1:] - crow[:-1])
        g_o["dvals"] = g_o["dGs"][row, col]
        g_o.pop("dGs")
    bad = []
    def chk(got, ref, what, atol_scale=1e-5):
        n, w = O.violations(got, ref, atol_scale=atol_scale)
        if n:
            bad.append(f"{what}: {n}/{ref.numel()} outside rtol 1e-4 + {atol_scale} mean|ref|, worst {w:.2e} x mean|ref|")
    chk(Hn, Hn_o, "Hn")
    for k in ("dXt", "dH"):
        chk(g[k], g_o[k], k)
    for k in REDUCED:
        if k in g:
            chk(g[k], g_o[k], k, 3e-5 if many else 1e-5)
    if many:
        floor = fp32_reference_floor(t, cfg)
        print(f"{name}: {rows} rows; fp32 reference vs fp64, worst x mean|ref|: "
              + ", ".join(f"{k} {w:.2e}" for k, w in floor.items()))
    assert not bad, f"{name} (B={cfg['B']}): " + "; ".join(bad)


@pytest.mark.parametrize("name", list(CASES))
def test_conv_variant_matches_oracle(name):
    spec = CASES[name]
    B = batch_of(spec)
    t, cfg, v, Hn, g, kernels = run_case(spec, B, seed=len(name) + 7 * spec["N"])
    check_kernels(name, spec["kernels"], kernels)
    compare_with_oracle(name, t, cfg, v, Hn, g, spec)
    if spec["B"] is None:   # batch independence: a sample of the big batch equals that sample run alone
        with torch.no_grad():
            for b in (0, B // 2, B - 1):
                one = dict(v)
                one["Xt"], one["H"] = v["Xt"][b:b + 1], v["H"][b:b + 1]
                alone = cell_step(one, spec)
                full = Hn[b].to(DEV)
                assert torch.allclose(alone[0], full, rtol=0, atol=1e-6), \
                    f"{name}: sample {b} alone differs from the batch by {(alone[0] - full).abs().max().item():.2e}"


# ---- the diagnostic switches, one fresh process each (every switch is read once per process) --------------------------
ARM_CASES = {"sf": "mt_sf_din16", "big": "h64_hout128", "kc3": "mt_kc3"}
ARMS = {
    "STC_DISABLE_TC=1": dict(env={"STC_DISABLE_TC": "1"}, kernels={
        "sf": {F_FF1, F_FF2, DX_FF1, DW_FF1}, "big": {F_FF2, DX_FF2, DW_FF2}, "kc3": {F_FF1, F_FF2, DX_FF1, DW_FF1}}),
    "STC_OPT=5": dict(env={"STC_OPT": "5"}, kernels={   # generic tensor-core epilogues
        "sf": {F_TC0, DX_GEN, DWP2, DWP4}, "big": {F_BIG, DX_BIG, DW_BIG}, "kc3": {F_TC0, DX_GEN, DWP4, DW_FF1}}),
    "STC_OPT=9": dict(env={"STC_OPT": "9"}, kernels={   # A operand staged in shared memory
        "sf": {F_TC1, F_TC2, DX_FAST, DWP2, DWP4}, "big": {F_BIG, DX_BIG, DW_BIG}, "kc3": {F_TC0, DX_FAST, DWP4, DW_FF1}}),
    "STC_OPT=33": dict(env={"STC_OPT": "33"}, kernels={  # wide-state dx (and so dW) on the general path
        "sf": SF_AT | {DWP2, DWP4}, "big": {F_BIG, DX_FF2, DW_FF2}, "kc3": {F_TC0, DX_FAST, DWP4, DW_FF1}}),
    "STC_DW_NO_PIPE=1": dict(env={"STC_DW_NO_PIPE": "1"}, kernels={
        "sf": SF_AT | {DW2, DW4}, "big": {F_BIG, DX_BIG, DW_BIG}, "kc3": {F_TC0, DX_FAST, DW4, DW_FF1}}),
}


def _arm_child(arm):
    """Body of the child process of test_diagnostic_switch: every arm case against the oracle and its forced kernels."""
    for short, name in ARM_CASES.items():
        spec = dict(CASES[name], kernels=frozenset(ARMS[arm]["kernels"][short]))
        B = batch_of(spec)
        t, cfg, v, Hn, g, kernels = run_case(spec, B, seed=11 + len(short))
        check_kernels(f"{arm} {name}", spec["kernels"], kernels)
        compare_with_oracle(f"{arm} {name}", t, cfg, v, Hn, g, spec)
        print(f"{arm} {name} B={B}: OK, ran {sorted(kernels)}", flush=True)


@pytest.mark.parametrize("arm", list(ARMS))
def test_diagnostic_switch(arm):
    env = {k: v for k, v in os.environ.items() if k not in ("STC_DISABLE_TC", "STC_OPT", "STC_DW_NO_PIPE")}
    env.update(ARMS[arm]["env"])
    code = f"import sys; sys.path.insert(0, {ROOT!r}); from tests.test_conv_variants_gpu import _arm_child; _arm_child({arm!r})"
    try:
        res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    except subprocess.TimeoutExpired as e:   # subprocess.run has killed and reaped the child
        pytest.fail(f"{arm}: child timed out after {e.timeout} s\n{(e.stdout or '')[-3000:]}")
    print(res.stdout[-3000:])
    assert res.returncode == 0, f"{arm}: child exited with {res.returncode}\n{res.stdout[-3000:]}\n{res.stderr[-5000:]}"


# ---- stack roll-outs against the fp64 oracle stack, on every tier the shared-terms fold runs on ------------------------
STACK_CASES = {
    "ffma_h7": dict(N=20, C=3, Din=2, h=7, Ks=2, Kc=2, B=3),           # FFMA dx fold
    "ffma_kc3": dict(N=20, C=4, Din=1, h=16, Ks=2, Kc=3, B=3),         # Kc = 3 (FFMA gates dW, tensor-core dx)
    "h8_split": dict(N=24, C=5, Din=1, h=8, Ks=2, Kc=2, B=3),          # candidate FFMA, gates tensor cores
    "big_h64": dict(N=16, C=4, Din=1, h=64, Ks=2, Kc=2, B=2),          # wide-state kernels
    "sf_multi_tile": dict(N=100, C=5, Din=1, h=16, Ks=2, Kc=2, B=None),
    "dense_ks3": dict(N=30, C=5, Din=1, h=16, Ks=3, Kc=2, B=3),
}
HOP_KINDS = ("tc_support", "tc_support_big", "support_dense", "support_csr")


def _stack_floor(got, ref, name, bad):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    err = (got - ref).abs()
    tol = 1e-4 * ref.abs() + 5e-5 * ref.abs().mean()
    n = int((err > tol).sum())
    if n:
        bad.append(f"{name}: {n}/{ref.numel()} outside the stack floor, worst {(err / ref.abs().mean()).max().item():.2e}"
                   " x mean|ref|")


@pytest.mark.parametrize("x_grad", [False, True], ids=["x_const", "x_grad"])
@pytest.mark.parametrize("name", list(STACK_CASES))
def test_stack_rollout_matches_oracle_stack(name, x_grad):
    import stc_gnn_b200 as S
    from stc_gnn_b200 import _lib
    from tests.test_shared_terms_gpu import reference_rollout
    p = STACK_CASES[name]
    N, C, Din, h, Ks, Kc = (p[k] for k in ("N", "C", "Din", "h", "Ks", "Kc"))
    B = p["B"] or multi_tile_batch(N, C, torch.cuda.get_device_properties(0).multi_processor_count)[0]
    layers, T, horizon = 2, 3, 2
    torch.manual_seed(len(name))
    stack = S.RecurrentStack(N, C, Ks, Kc, Din, h, layers, horizon).to(DEV)
    g = torch.Generator().manual_seed(len(name) + 1)
    Gs0 = (torch.rand(N, N, generator=g) * (2.0 / N)).float()
    Gc0 = (torch.rand(C, C, generator=g) * (2.0 / C)).float()
    X0 = (torch.rand(B, T, N, C, Din, generator=g) < 0.3).float()
    dOut = torch.randn(B, horizon, N, C, h, generator=g).float()
    Gs, Gc = Gs0.to(DEV).requires_grad_(True), Gc0.to(DEV).requires_grad_(True)
    X = X0.to(DEV).requires_grad_(x_grad)
    leaves = list(stack.parameters()) + [Gs, Gc] + ([X] if x_grad else [])

    def step(fn):
        for t_ in leaves:
            t_.grad = None
        _lib.timing_enable(True)
        _lib.timing_collect()
        out = fn()
        out.backward(dOut.to(DEV))
        torch.cuda.synchronize()
        _lib.timing_enable(False)
        hops = sum(v[1] for k, v in _lib.timing_collect().items() if k in HOP_KINDS)
        return out.detach().clone(), [t_.grad.clone() for t_ in leaves], hops

    out_r, _, hops_r = step(lambda: reference_rollout(stack, Gs, Gc, X))
    out, grads, hops = step(lambda: stack(Gs, Gc, X))
    assert hops < hops_r, f"{name}: the stack launched {hops} spatial hops, the unshared roll-out {hops_r}: nothing shared"
    assert torch.equal(out, out_r), f"{name}: the shared forward is not bitwise the unshared one"
    # fp64 oracle stack
    cells = [O.CellParams(*(getattr(getattr(c, conv), pn).detach().double().cpu().requires_grad_(True)
                            for conv, pn in (("gates", "W"), ("gates", "b"), ("candi", "W"), ("candi", "b"))))
             for c in list(stack.encoder) + list(stack.decoder)]
    Gs_o, Gc_o = Gs0.double().requires_grad_(True), Gc0.double().requires_grad_(True)
    X_o = X0.double().requires_grad_(x_grad)
    ref = O.stack_forward(Gs_o, Gc_o, X_o, cells[:layers], cells[layers:], horizon, Ks, Kc)
    ref.backward(dOut.double())
    bad = []
    O.assert_close(out.cpu(), ref.detach(), f"{name} stack out")
    names = [n for n, _ in stack.named_parameters()]
    ref_grads = [getattr(c, a).grad for c in cells for a in ("Wg", "bg", "Wc", "bc")] + [Gs_o.grad, Gc_o.grad] + \
        ([X_o.grad] if x_grad else [])
    for nm, got, r in zip(names + ["Gs", "Gc"] + (["X_seq"] if x_grad else []), grads, ref_grads):
        _stack_floor(got, r, nm, bad)
    assert not bad, f"{name} (B={B}, x_grad={x_grad}): " + "; ".join(bad)
