"""ctypes binding of the C-ABI library (include/vorta_b200.h).

The library is built in-tree by ``vorta_b200/csrc/Makefile`` (``__graft_entry__.build()``).  There is no
fallback: if the shared object is missing, or a compute entry point is called without a B200, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VB_LIB_PATH") or os.path.join(_HERE, "lib", "libvorta_b200.so")   # override: perf experiments
CSRC_DIR = os.path.join(_HERE, "csrc")

VB_OK = 0
VB_ERR_INVALID = -1
VB_ERR_CUDA = -2
VB_ERR_UNSUPPORTED = -3

BRANCH_FULL, BRANCH_CORESET, BRANCH_SLIDING, BRANCH_SKIP = 0, 1, 2, -1
BRANCH_FULL_LO, BRANCH_FULL_HI = 3, 4          # full attention over the lower / upper half of the query work items
DTYPE_F32, DTYPE_BF16 = 0, 1
ATTN_CORESET_KV_FROM_K = 1


def branch_full_part(k: int, n: int) -> int:
    """VB_BRANCH_FULL_PART(k, n): full attention over part k of n equal parts of the query work items."""
    return 16 + 8 * n + k


# vb_plan_query keys
(PLAN_SEQ_LEN, PLAN_NUM_GROUPS, PLAN_GROUP_SIZE, PLAN_CORESET_LEN, PLAN_NUM_TILES, PLAN_TILE_TOKENS,
 PLAN_NUM_POOLED, PLAN_KEYS_PER_QUERY, PLAN_SLIDING_PAIRS, PLAN_SLIDING_RUNS) = range(10)
# vb_plan_export keys
(EXPORT_CENTER_INDICES, EXPORT_MARGIN_INDICES, EXPORT_TILE_MAP, EXPORT_TILE_WINDOW, EXPORT_SLIDING_RUNS,
 EXPORT_SLIDING_ITEMS, EXPORT_SLIDING_QUERY_MAP) = range(7)

# every symbol include/vorta_b200.h declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = (
    "vb_last_error", "vb_version", "vb_device_check",
    "vb_plan_create", "vb_plan_destroy", "vb_plan_set_text_valid", "vb_plan_query", "vb_plan_export",
    "vb_router_forward", "vb_coreset_select", "vb_coreset_tables", "vb_gather_rows",
    "vb_attn_workspace_bytes", "vb_attn_fwd", "vb_attn_dense",
    "vb_block_ln_modulate", "vb_block_gate_residual", "vb_block_rmsnorm_rope", "vb_block_headnorm_rope",
    "vb_stats_reset", "vb_stats_launches", "vb_stats_attn_flops", "vb_timing_enable", "vb_timing_collect",
    "vb_timing_collect_kinds",
    "vb_ulysses_pack_heads", "vb_ulysses_pack_qkv", "vb_ulysses_unpack_heads", "vb_ulysses_scatter_qkv_slots",
)


class PlanDesc(C.Structure):
    _fields_ = [
        ("latent", C.c_int32 * 3),
        ("tile", C.c_int32 * 3),
        ("window", C.c_int32 * 3),
        ("lowres_window", C.c_int32 * 3),
        ("n_unpooled", C.c_int32),
        ("text_len", C.c_int32),
        ("text_valid", C.c_int32),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p),
        ("q_stride", C.c_int64 * 3), ("k_stride", C.c_int64 * 3),
        ("v_stride", C.c_int64 * 3), ("out_stride", C.c_int64 * 3),
        ("batch", C.c_int32), ("heads", C.c_int32),
        ("branch", C.POINTER(C.c_int32)),
        ("weights", C.POINTER(C.c_float)),
        ("flags", C.c_uint32),
        ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_int64),
        ("debug", C.c_void_p),
        ("out_peer_ptrs", C.c_void_p * 8),
        ("out_peer_count", C.c_int32),
        ("out_peer_rows", C.c_int32),
        ("out_heads", C.POINTER(C.c_int32)),
        ("weights_device", C.c_void_p),
        ("text_valid", C.POINTER(C.c_int32)),
    ]


class VortaB200Error(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def build(verbose: bool = False) -> str:
    """Compile the shared library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    res = subprocess.run(["make", "-C", CSRC_DIR], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0:
        raise VortaB200Error(f"building {LIB_PATH} failed (exit {res.returncode})")
    return LIB_PATH


def _declare(lib: C.CDLL) -> None:
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    lib.vb_last_error.restype = C.c_char_p
    lib.vb_last_error.argtypes = []
    lib.vb_version.restype = C.c_int
    lib.vb_device_check.restype = C.c_int
    lib.vb_plan_create.restype = C.c_int
    lib.vb_plan_create.argtypes = [C.POINTER(vp), C.POINTER(PlanDesc)]
    lib.vb_plan_destroy.restype = None
    lib.vb_plan_destroy.argtypes = [vp]
    lib.vb_plan_set_text_valid.restype = C.c_int
    lib.vb_plan_set_text_valid.argtypes = [vp, i32]
    lib.vb_plan_query.restype = C.c_int
    lib.vb_plan_query.argtypes = [vp, C.c_int, C.POINTER(i64)]
    lib.vb_plan_export.restype = C.c_int
    lib.vb_plan_export.argtypes = [vp, C.c_int, vp, C.POINTER(i64)]
    lib.vb_router_forward.restype = C.c_int
    lib.vb_router_forward.argtypes = [vp, C.c_int, vp, vp, C.c_int, i64, i64, i32, i32, i32, i32, f32, vp, vp, vp]
    lib.vb_coreset_select.restype = C.c_int
    lib.vb_coreset_select.argtypes = [vp, vp, i64, i64, i64, i32, i32, vp, vp, vp, vp, vp]
    lib.vb_coreset_tables.restype = C.c_int
    lib.vb_coreset_tables.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp, vp]
    lib.vb_attn_dense.restype = C.c_int
    lib.vb_attn_dense.argtypes = [vp, vp, vp, vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64),
                                  i32, i32, i32, i32, vp]
    lib.vb_gather_rows.restype = C.c_int
    lib.vb_gather_rows.argtypes = [vp, i64, i64, i64, vp, i64, i64, i64, vp, i64, i64, i32, i32, i32, vp]
    lib.vb_attn_workspace_bytes.restype = i64
    lib.vb_attn_workspace_bytes.argtypes = [vp, i32, i32]
    lib.vb_attn_fwd.restype = C.c_int
    lib.vb_attn_fwd.argtypes = [vp, C.POINTER(AttnArgs), vp]
    lib.vb_stats_reset.restype = None
    lib.vb_stats_launches.restype = i64
    lib.vb_stats_attn_flops.restype = C.c_double
    lib.vb_block_ln_modulate.restype = C.c_int
    lib.vb_block_ln_modulate.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, i32, f32, vp]
    lib.vb_block_gate_residual.restype = C.c_int
    lib.vb_block_gate_residual.argtypes = [vp, vp, vp, vp, i64, i32, i32, vp]
    lib.vb_block_rmsnorm_rope.restype = C.c_int
    lib.vb_block_rmsnorm_rope.argtypes = [vp, vp, vp, vp, vp, i64, i32, i32, f32, vp]
    lib.vb_block_headnorm_rope.restype = C.c_int
    lib.vb_block_headnorm_rope.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, f32, vp]
    lib.vb_timing_enable.restype = None
    lib.vb_timing_enable.argtypes = [C.c_int]
    lib.vb_timing_collect.restype = C.c_int
    lib.vb_timing_collect.argtypes = [C.POINTER(C.c_double), C.POINTER(i64), C.POINTER(C.c_double)]
    lib.vb_timing_collect_kinds.restype = C.c_int
    lib.vb_timing_collect_kinds.argtypes = [C.POINTER(C.c_double), C.POINTER(i64), C.POINTER(C.c_double)]
    lib.vb_ulysses_pack_heads.restype = C.c_int
    lib.vb_ulysses_pack_heads.argtypes = [vp, vp, i32, i32, i32, i32, i64, i64, C.POINTER(i32), vp]
    lib.vb_ulysses_pack_qkv.restype = C.c_int
    lib.vb_ulysses_pack_qkv.argtypes = [vp, vp, vp, C.POINTER(i64), C.POINTER(i64), vp, i32, i32, i32, C.POINTER(i32), vp]
    lib.vb_ulysses_scatter_qkv_slots.restype = C.c_int
    lib.vb_ulysses_scatter_qkv_slots.argtypes = [vp, vp, vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(vp), i64, i32, i32,
                                                 i32, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), i32, vp]
    lib.vb_ulysses_unpack_heads.restype = C.c_int
    lib.vb_ulysses_unpack_heads.argtypes = [vp, vp, i32, i32, i32, C.POINTER(i32), vp]


def lib() -> C.CDLL:
    """Load (once) and return the C-ABI library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VortaB200Error(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(vorta_b200 has no fallback path)")
        handle = C.CDLL(LIB_PATH)
        _declare(handle)
        _lib = handle
    return _lib


def check(rc: int) -> None:
    """Map a C-ABI return code to the exception type the reference raises for the same condition."""
    if rc == VB_OK:
        return
    msg = lib().vb_last_error().decode("utf-8", "replace")
    if rc == VB_ERR_INVALID:
        raise ValueError(msg)                      # reference: _check_input (vorta/attention/wan.py:181-193)
    raise VortaB200Error(f"vorta_b200 error {rc}: {msg}")
