"""The C-ABI library loads and exports every symbol include/vorta_b200.h declares (no compute calls: CPU-only)."""
import ctypes
import os
import re

import pytest

from vorta_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "vorta_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = L.lib()
    declared = _declared_symbols()
    assert len(declared) >= 20
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in the header but not exported"
    assert sorted(L.EXPORTED_SYMBOLS) == declared


def test_header_is_plain_c():
    # the boundary must not leak C++ / torch types
    text = open(os.path.join(ROOT, "include", "vorta_b200.h")).read()
    assert 'extern "C"' in text
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)      # comments may mention torch; declarations may not
    for banned in ("std::", "torch", "at::Tensor", "template", "class "):
        assert banned not in text


def test_version_and_error_string():
    lib = L.lib()
    assert lib.vb_version() >= 100
    assert isinstance(lib.vb_last_error(), bytes)


def test_invalid_plan_is_value_error_with_reference_message():
    from vorta_b200 import ops
    # reference: wan.py:186-189
    with pytest.raises(ValueError, match=r"Tile size \(5, 9, 8\) \(dim=5\) does not divide latent shape \(21, 45, 80\)"):
        ops.Plan((21, 45, 80), (5, 9, 8), (3, 3, 3), (3, 3, 2))
    # reference: wan.py:191-193
    with pytest.raises(ValueError, match=r"does not match low-res info"):
        ops.Plan((21, 45, 80), (3, 9, 16), (3, 3, 3), (2, 3, 2))


def test_no_cuda_means_loud_failure():
    import torch
    from vorta_b200 import ops
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    plan = ops.Plan((4, 6, 4), (2, 3, 2), (3, 3, 3), (2, 3, 2))
    x = torch.zeros(1, 1, 96, 128, dtype=torch.bfloat16)
    with pytest.raises(L.VortaB200Error):
        ops.routed_attention(plan, x, x, x, branch=[0])
    with pytest.raises(L.VortaB200Error):
        ops.coreset_select(plan, x)
    assert L.lib().vb_device_check() == L.VB_ERR_UNSUPPORTED


def test_block_kernels_refuse_misaligned_vector_pointers():
    """Every pointer a block kernel reads or writes with 16-byte vectors must be 16-byte aligned: VB_ERR_INVALID is
    returned before any launch (the addresses below are never dereferenced)."""
    lib = L.lib()
    A, M = 0x10000, 0x10008                    # aligned, misaligned (8 bytes past a 16-byte boundary)
    rows, dim = 4, 1536
    for x, out in ((M, A), (A, M)):
        assert lib.vb_block_ln_modulate(x, None, None, None, None, out, rows, dim, rows, 1e-6, None) == L.VB_ERR_INVALID
        assert lib.vb_block_rmsnorm_rope(x, A, None, None, out, rows, dim, rows, 1e-6, None) == L.VB_ERR_INVALID
    for x, y, out in ((M, A, A), (A, M, A), (A, A, M)):
        assert lib.vb_block_gate_residual(x, y, None, out, rows, dim, rows, None) == L.VB_ERR_INVALID
    assert lib.vb_block_rmsnorm_rope(A, M, None, None, A, rows, dim, rows, 1e-6, None) == L.VB_ERR_INVALID
    hn = (lambda x, w, c, s, out: lib.vb_block_headnorm_rope(x, w, c, s, out, 1, rows, 12, rows, rows, 0, 1e-6, None))
    for args in ((M, A, A, A, A), (A, M, A, A, A), (A, A, M, A, A), (A, A, A, M, A), (A, A, A, A, M),
                 (A, None, M, A, A)):
        assert hn(*args) == L.VB_ERR_INVALID, args
    assert b"16-byte" in lib.vb_last_error()
