"""ctypes binding of libstc_b200.so -- the C ABI declared in include/stc_b200.h.

The product path has no CPU fallback: if the library cannot be loaded, or a call returns a negative
status, a RuntimeError carrying stc_last_error() is raised.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libstc_b200.so")

ABI_VERSION = 7
ACT_NONE, ACT_RELU = 0, 1
SUPPORT_DENSE, SUPPORT_CSR = 0, 1

# every symbol include/stc_b200.h declares (tests check the built library exports all of them)
EXPORTED = (
    "stc_abi_version", "stc_last_error", "stc_cell_saved_bytes", "stc_cell_bwd_scratch_bytes",
    "stc_cell_fwd", "stc_cell_bwd", "stc_support_apply", "stc_last_launch_count",
    "stc_timing_enable", "stc_timing_collect", "stc_kernel_kind_name", "stc_tf32x3_gemm",
    "stc_cell_saved_layout", "stc_cell_fwd_stage", "stc_debug_trace_set",
    "stc_cell_bwd_scratch_layout", "stc_cell_bwd_stage",
    "stc_support_apply_rows", "stc_halo_pack", "stc_halo_unpack", "stc_concurrency_set",
    "stc_cell_fwd_x", "stc_cell_bwd_x", "stc_support_outer", "stc_support_apply_edge_grad",
    "stc_support_apply_rows_edge_grad", "stc_pair_scores_csr", "stc_edge_softmax_fwd", "stc_edge_softmax_bwd",
    "stc_pair_scores_csr_rows", "stc_pair_topk_workspace_bytes", "stc_pair_topk",
    "stc_pair_topk_rows_workspace_bytes", "stc_pair_topk_rows",
)
STAGE_GATES, STAGE_CANDI = 0, 1
SAVED_REGIONS = ("u", "r", "c", "Yr", "Yx", "Yh", "Q", "Pg", "Pc")
SCRATCH_REGIONS = ("dYr", "dYx", "dYh")


class StcDims(Structure):
    _fields_ = [(n, c_int32) for n in ("B", "N", "C", "Din", "h", "Ks", "Kc", "act", "has_bias")]


class StcSupport(Structure):
    _fields_ = [("kind", c_int32), ("nnz", c_int64), ("vals", c_void_p), ("rowptr", c_void_p), ("col", c_void_p),
                ("t_vals", c_void_p), ("t_rowptr", c_void_p), ("t_col", c_void_p)]


_lib = None


def load(build_if_missing: bool = True):
    """Load (building first if the sources changed and nvcc is present) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        from .build import build
        build()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -m stc_gnn_b200.build` (no CPU fallback exists)")
    lib = ctypes.CDLL(LIB_PATH)
    lib.stc_abi_version.restype = c_int
    lib.stc_last_error.restype = c_char_p
    lib.stc_last_launch_count.restype = c_int
    lib.stc_cell_saved_bytes.restype = c_size_t
    lib.stc_cell_saved_bytes.argtypes = [POINTER(StcDims)]
    lib.stc_cell_bwd_scratch_bytes.restype = c_size_t
    lib.stc_cell_bwd_scratch_bytes.argtypes = [POINTER(StcDims)]
    lib.stc_cell_fwd.restype = c_int
    lib.stc_cell_fwd.argtypes = [POINTER(StcDims), POINTER(StcSupport), c_void_p, c_void_p, c_int64, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.stc_cell_fwd_x.restype = c_int
    lib.stc_cell_fwd_x.argtypes = lib.stc_cell_fwd.argtypes[:-1] + [c_void_p, c_void_p, c_void_p]
    lib.stc_support_outer.restype = c_int
    lib.stc_support_outer.argtypes = [c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p, c_float, c_void_p, c_void_p]
    lib.stc_support_apply_edge_grad.restype = c_int
    lib.stc_support_apply_edge_grad.argtypes = [POINTER(StcSupport), c_int32, c_int32, c_int32, c_void_p, c_int64,
                                                c_void_p, c_int64, c_void_p, c_float, c_float, c_void_p, c_int64,
                                                c_float, c_void_p, c_void_p]
    lib.stc_support_apply_rows_edge_grad.restype = c_int
    lib.stc_support_apply_rows_edge_grad.argtypes = lib.stc_support_apply_edge_grad.argtypes[:-1] + [c_void_p, c_int32,
                                                                                                    c_void_p]
    lib.stc_pair_scores_csr.restype = c_int
    lib.stc_pair_scores_csr.argtypes = [POINTER(StcSupport), c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.stc_pair_scores_csr_rows.restype = c_int
    lib.stc_pair_scores_csr_rows.argtypes = [POINTER(StcSupport), c_int32, c_int64, c_int64, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_int32, c_void_p]
    lib.stc_pair_topk_workspace_bytes.restype = c_size_t
    lib.stc_pair_topk_workspace_bytes.argtypes = [c_int32, c_int64, c_int32]
    lib.stc_pair_topk.restype = c_int
    lib.stc_pair_topk.argtypes = [c_int32, c_int64, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_size_t,
                                  c_void_p]
    lib.stc_pair_topk_rows_workspace_bytes.restype = c_size_t
    lib.stc_pair_topk_rows_workspace_bytes.argtypes = [c_int32, c_int64, c_int32, c_int32]
    lib.stc_pair_topk_rows.restype = c_int
    lib.stc_pair_topk_rows.argtypes = [c_int32, c_int64, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p,
                                       c_void_p, c_void_p, c_size_t, c_void_p]
    lib.stc_edge_softmax_fwd.restype = c_int
    lib.stc_edge_softmax_fwd.argtypes = [POINTER(StcSupport), c_int32, c_void_p, c_void_p, c_void_p]
    lib.stc_edge_softmax_bwd.restype = c_int
    lib.stc_edge_softmax_bwd.argtypes = [POINTER(StcSupport), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.stc_cell_saved_layout.restype = c_int
    lib.stc_cell_saved_layout.argtypes = [POINTER(StcDims), POINTER(c_int64), c_int32]
    lib.stc_cell_fwd_stage.restype = c_int
    lib.stc_cell_fwd_stage.argtypes = [POINTER(StcDims), c_int32, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.stc_cell_bwd.restype = c_int
    lib.stc_cell_bwd.argtypes = [POINTER(StcDims), POINTER(StcSupport), c_void_p, c_void_p, c_int64, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_size_t, c_void_p, c_size_t,
                                 c_void_p]
    lib.stc_cell_bwd_x.restype = c_int
    lib.stc_cell_bwd_x.argtypes = lib.stc_cell_bwd.argtypes[:-1] + [c_void_p] * 7
    lib.stc_cell_bwd_scratch_layout.restype = c_int
    lib.stc_cell_bwd_scratch_layout.argtypes = [POINTER(StcDims), POINTER(c_int64), c_int32]
    lib.stc_cell_bwd_stage.restype = c_int
    lib.stc_cell_bwd_stage.argtypes = [POINTER(StcDims), c_int32, c_void_p, c_void_p, c_int64, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_int32, c_void_p, c_size_t, c_void_p, c_size_t, c_void_p]
    lib.stc_support_apply.restype = c_int
    lib.stc_support_apply.argtypes = [POINTER(StcSupport), c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64,
                                      c_void_p, c_int64, c_void_p, c_float, c_float, c_void_p]
    lib.stc_support_apply_rows.restype = c_int
    lib.stc_support_apply_rows.argtypes = [POINTER(StcSupport), c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64,
                                           c_void_p, c_int64, c_void_p, c_float, c_float, c_void_p, c_int32, c_void_p]
    lib.stc_halo_pack.restype = c_int
    lib.stc_halo_pack.argtypes = [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p]
    lib.stc_halo_unpack.restype = c_int
    lib.stc_halo_unpack.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p]
    lib.stc_concurrency_set.restype = c_int
    lib.stc_concurrency_set.argtypes = [c_int32]
    lib.stc_tf32x3_gemm.restype = c_int
    lib.stc_tf32x3_gemm.argtypes = [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p]
    lib.stc_timing_enable.restype = c_int
    lib.stc_timing_enable.argtypes = [c_int32]
    lib.stc_timing_collect.restype = c_int
    lib.stc_timing_collect.argtypes = [POINTER(ctypes.c_double), POINTER(c_int64), POINTER(ctypes.c_double), c_int32]
    lib.stc_debug_trace_set.restype = c_int
    lib.stc_debug_trace_set.argtypes = [c_void_p, c_int64]
    lib.stc_kernel_kind_name.restype = c_char_p
    lib.stc_kernel_kind_name.argtypes = [c_int32]
    if lib.stc_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libstc_b200.so ABI {lib.stc_abi_version()} != binding ABI {ABI_VERSION}: rebuild")
    _lib = lib
    return lib


def saved_layout(dims: StcDims) -> dict:
    """{region name: offset in floats} of the `saved` buffer of one cell call."""
    lib = load()
    offs = (c_int64 * len(SAVED_REGIONS))()
    check(lib.stc_cell_saved_layout(dims, offs, len(SAVED_REGIONS)), "stc_cell_saved_layout")
    return {n: int(offs[i]) for i, n in enumerate(SAVED_REGIONS)}


def scratch_layout(dims: StcDims) -> dict:
    """{region name: offset in floats} of the adjoint regions of the backward `scratch` buffer."""
    lib = load()
    offs = (c_int64 * len(SCRATCH_REGIONS))()
    check(lib.stc_cell_bwd_scratch_layout(dims, offs, len(SCRATCH_REGIONS)), "stc_cell_bwd_scratch_layout")
    return {n: int(offs[i]) for i, n in enumerate(SCRATCH_REGIONS)}


def check(status: int, what: str) -> None:
    if status != 0:
        msg = _lib.stc_last_error().decode("utf-8", "replace") if _lib is not None else ""
        raise RuntimeError(f"{what} failed (status {status}): {msg}")


def last_launch_count() -> int:
    return int(load().stc_last_launch_count())


# running total of kernels launched through the library by this process (bench.py's gpu_launches)
LAUNCHES = 0


def note_launches() -> None:
    global LAUNCHES
    LAUNCHES += int(_lib.stc_last_launch_count())


def set_concurrency(mode: int) -> None:
    """-1: fork independent kernels of a cell call onto side streams only for small problems (default); 0: never; 1: always."""
    check(load().stc_concurrency_set(int(mode)), "stc_concurrency_set")


def timing_enable(on: bool) -> None:
    load().stc_timing_enable(1 if on else 0)


def timing_collect():
    """{kernel kind: (device ms, launches, algorithmic bytes)} since the last collect."""
    lib = load()
    n = 32
    ms = (ctypes.c_double * n)()
    cnt = (c_int64 * n)()
    by = (ctypes.c_double * n)()
    kinds = lib.stc_timing_collect(ms, cnt, by, n)
    return {lib.stc_kernel_kind_name(k).decode(): (ms[k], int(cnt[k]), by[k]) for k in range(kinds) if cnt[k]}
