"""Fused elementwise kernels of the DiT block (SURVEY.md section 8f rows 1-2) against fp64 references of the same op,
held to the bar derived in test_block_numerics.py: half a bf16 ulp of the fp64 result plus twice the kernel's fp32 error
bound.  Every dispatch instance runs: the warp-per-row kernels at all seven widths (1024 to 6144 channels, 1, 2 and 4
warps per row, every tail of a CTA's rows), the CTA-per-row fallback at other widths and, through the C ABI with a
misaligned fp32 parameter (which the dispatcher sends to the fallback), at the production widths; output buffers are
fenced with NaN guard rows that must stay untouched bit for bit."""
import math
import zlib

import numpy as np
import pytest
import torch

from vorta_b200 import _lib as L
from vorta_b200 import ops

from test_block_numerics import (HEAD, WARP_DIMS, bf16_values, check_bar, check_bias, gate_ref, headnorm_ref,
                                 ln_ref, rms_ref, rows_per_cta)

pytestmark = pytest.mark.gpu

NAN16 = 0x7FC1                   # a bf16 NaN bit pattern no kernel produces


def _np(t):
    return t.detach().float().cpu().numpy().astype(np.float64)


def _bf16(a):
    return torch.from_numpy(np.asarray(a, np.float32)).to(torch.bfloat16).cuda()


def _f32(a):
    return torch.from_numpy(np.asarray(a, np.float32)).cuda()


def _misaligned(a):
    """fp32 copy of a that starts 4 bytes past a 16-byte boundary (scalar loads only: the fallback kernels)."""
    a = np.asarray(a, np.float32)
    buf = torch.empty(a.size + 4, dtype=torch.float32, device="cuda")
    v = buf[1:1 + a.size].view(a.shape)
    v.copy_(torch.from_numpy(a))
    assert v.data_ptr() % 16 == 4
    return v


def _fenced(rows, dim, guard=3):
    """A bf16 buffer of rows + 2 guard rows of NaN bits; returns (buffer, view of the middle rows)."""
    buf = torch.full(((rows + 2 * guard) * dim,), NAN16, dtype=torch.int16, device="cuda").view(torch.bfloat16)
    return buf, buf[guard * dim:(guard + rows) * dim].view(rows, dim)


def _guards_intact(buf, rows, dim, guard=3):
    bits = buf.view(torch.int16)
    head, tail = bits[:guard * dim], bits[(guard + rows) * dim:]
    return bool((head == NAN16).all()) and bool((tail == NAN16).all())


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _abi_ln(x, w, b, sc, sh, out, rows_per_batch, eps=1e-6):
    rows, dim = out.shape
    L.check(L.lib().vb_block_ln_modulate(x.data_ptr(), _ptr(w), _ptr(b), _ptr(sc), _ptr(sh), out.data_ptr(), rows, dim,
                                         rows_per_batch, eps, torch.cuda.current_stream().cuda_stream))


def _abi_rms(x, w, cos, sin, out, tokens_per_batch, eps=1e-6):
    rows, dim = out.shape
    L.check(L.lib().vb_block_rmsnorm_rope(x.data_ptr(), w.data_ptr(), _ptr(cos), _ptr(sin), out.data_ptr(), rows, dim,
                                          tokens_per_batch, eps, torch.cuda.current_stream().cuda_stream))


def run_ln(x, w=None, b=None, sc=None, sh=None, rows_per_batch=None, fallback=False, eps=1e-6):
    """numpy in, numpy out: ops.ln_modulate, or the ABI with misaligned fp32 parameters (the CTA-per-row kernel) and a
    fenced output.  With no parameter at all the fallback gets a misaligned weight of ones (t * 1 + 0 is exact)."""
    rows, dim = x.shape
    rpb = rows if rows_per_batch is None else rows_per_batch
    xt = _bf16(x)
    if not fallback:
        B = rows // rpb
        out = ops.ln_modulate(xt.view(B, rpb, dim), None if w is None else _f32(w), None if b is None else _f32(b),
                              None if sc is None else _f32(sc), None if sh is None else _f32(sh), eps)
        return _np(out.view(rows, dim))
    if w is None and b is None and sc is None:
        w = np.ones(dim, np.float32)
    buf, out = _fenced(rows, dim)
    m = lambda a: None if a is None else _misaligned(a)
    _abi_ln(xt, m(w), m(b), m(sc), m(sh), out, rpb, eps)
    torch.cuda.synchronize()
    assert _guards_intact(buf, rows, dim)
    return _np(out)


def run_rms(x, w, cos=None, sin=None, tokens_per_batch=None, fallback=False, eps=1e-6):
    """ops.rmsnorm_rope, or the ABI with misaligned fp32 tables (the CTA-per-row kernel) and a fenced output."""
    rows, dim = x.shape
    tpb = rows if tokens_per_batch is None else tokens_per_batch
    xt, wt = _bf16(x), _bf16(w)
    if not fallback:
        out = ops.rmsnorm_rope(xt.view(rows // tpb, tpb, dim), wt, eps, None if cos is None else _f32(cos),
                               None if sin is None else _f32(sin))
        return _np(out.view(rows, dim))
    assert cos is not None
    buf, out = _fenced(rows, dim)
    _abi_rms(xt, wt, _misaligned(cos), _misaligned(sin), out, tpb, eps)
    torch.cuda.synchronize()
    assert _guards_intact(buf, rows, dim)
    return _np(out)


def _rng(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def _rows(rng, rows, dim, offset=0.0, std=1.0):
    return bf16_values(rng.standard_normal((rows, dim)) * std + offset)


def _tables(rng, tokens, exact=False):
    if exact:                                  # angles 0, pi/2, pi, 3pi/2 with exact table entries
        k = rng.integers(0, 4, (tokens, HEAD // 2))
        return np.choose(k, [1, 0, -1, 0]).astype(np.float32), np.choose(k, [0, 1, 0, -1]).astype(np.float32)
    ang = rng.random((tokens, HEAD // 2)) * 2 * math.pi
    return np.cos(ang).astype(np.float32), np.sin(ang).astype(np.float32)


# every dispatch instance: (dim, fallback)
LN_DISPATCH = ([(d, False) for d in WARP_DIMS] + [(d, True) for d in (1536, 3072, 5120)]
               + [(384, False), (640, False), (8192, False)])
_ids = [f"{d}-{'fallback' if fb else 'dispatch'}" for d, fb in LN_DISPATCH]


@pytest.mark.parametrize("B,S,dim", [(1, 333, 1536), (2, 130, 5120), (1, 64, 384), (1, 71, 3072), (2, 9, 2048),
                                     (1, 40, 1024), (2, 33, 4096), (1, 21, 6144), (2, 17, 640), (1, 9, 8192)])
def test_ln_modulate(B, S, dim):
    rng = _rng("ln", B, S, dim)
    x = _rows(rng, B * S, dim, 0.3, 2.0)
    sc, sh = (rng.standard_normal((2, B, dim)) * 0.2).astype(np.float32)
    w = (1 + 0.1 * rng.standard_normal(dim)).astype(np.float32)
    b = (0.1 * rng.standard_normal(dim)).astype(np.float32)
    for kw in (dict(sc=sc, sh=sh), dict(w=w, b=b), dict(), dict(w=w, b=b, sc=sc, sh=sh)):
        out = run_ln(x, rows_per_batch=S, **kw)
        ref = ln_ref(x, kw.get("w"), kw.get("b"), kw.get("sc"), kw.get("sh"), rows_per_batch=S)
        check_bar(out, ref, str(sorted(kw)))
        check_bias(out, ref[0], str(sorted(kw)))


@pytest.mark.parametrize("dim,fallback", LN_DISPATCH, ids=_ids)
def test_ln_modulate_mean_over_std(dim, fallback):
    """|mean| / std from 0 to 200 (bf16 resolves no more): the one-pass variance of the old fallback fails at 200."""
    rng = _rng("mean", dim, fallback)
    for offset in (0.0, 1.0, 16.0, 64.0, 200.0, -200.0):
        x = _rows(rng, 24, dim, offset)
        check_bar(run_ln(x, fallback=fallback), ln_ref(x, fallback=fallback), f"offset {offset}")


@pytest.mark.parametrize("dim,fallback", LN_DISPATCH, ids=_ids)
def test_ln_modulate_edges(dim, fallback):
    """Variance ~ eps, values around 1e4, constant rows (exactly bf16(shift)), all four parameters, bias alone."""
    rng = _rng("edges", dim, fallback)
    for what, x in (("var ~ eps", _rows(rng, 8, dim, 0.0, 1e-3)), ("1e4", _rows(rng, 8, dim, 0.0, 1e4)),
                    ("1e4 offset", _rows(rng, 8, dim, 1e4, 300.0))):
        check_bar(run_ln(x, fallback=fallback), ln_ref(x, fallback=fallback), what)
    rows = 10
    x = np.repeat(bf16_values(rng.standard_normal((rows, 1))), dim, 1)
    sc = (rng.standard_normal((2, dim)) * 0.2).astype(np.float32)
    g = rng.standard_normal((2, dim))
    sh = bf16_values(np.sign(g) * (0.5 + np.abs(g))).astype(np.float32)          # bf16 values, |shift| >= 1/2
    out = run_ln(x, sc=sc, sh=sh, rows_per_batch=rows // 2, fallback=fallback)
    assert np.array_equal(out, np.repeat(sh.astype(np.float64), rows // 2, 0)), "constant row -> bf16(shift)"
    x = _rows(rng, rows, dim, 0.5, 2.0)
    w = (1 + 0.1 * rng.standard_normal(dim)).astype(np.float32)
    b = (0.1 * rng.standard_normal(dim)).astype(np.float32)
    kw = dict(w=w, b=b, sc=sc, sh=sh)
    check_bar(run_ln(x, **kw, rows_per_batch=rows // 2, fallback=fallback),
              ln_ref(x, w, b, sc, sh, rows_per_batch=rows // 2, fallback=fallback), "weight, bias, scale, shift")
    # cancellation: shift ~ -t (1 + scale)
    t, _ = ln_ref(x[:1])
    sh1 = (-(t * (1 + sc[:1])) + rng.standard_normal((1, dim)) * 1e-3).astype(np.float32)
    check_bar(run_ln(x[:1], sc=sc[:1], sh=sh1, fallback=fallback), ln_ref(x[:1], None, None, sc[:1], sh1,
                                                                           fallback=fallback), "shift ~ -t(1+scale)")


@pytest.mark.parametrize("dim,fallback", LN_DISPATCH, ids=_ids)
def test_ln_modulate_bias_without_weight(dim, fallback):
    """LayerNorm(x) + bias with no weight, as F.layer_norm(x, shape, None, bias) computes it."""
    rng = _rng("bias", dim, fallback)
    x = _rows(rng, 6, dim, 0.3)
    b = (0.5 * rng.standard_normal(dim)).astype(np.float32)
    check_bar(run_ln(x, b=b, fallback=fallback), ln_ref(x, None, b, fallback=fallback), "bias without weight")
    if not fallback:
        xt = _bf16(x).view(1, 6, dim)
        want = torch.nn.functional.layer_norm(xt.double(), (dim,), None, _f32(b).double(), 1e-6)
        got = ops.ln_modulate(xt, None, _f32(b), None, None, 1e-6)
        check_bar(_np(got.view(6, dim)), (_np(want.view(6, dim)), ln_ref(x, None, b)[1]), "against F.layer_norm")


@pytest.mark.parametrize("dim", [1024, 2048, 4096, 1536, 3072, 6144])
def test_row_kernels_every_tail_and_fences(dim):
    """Row counts leaving 1 .. rows-per-CTA - 1 rows in the last CTA (whose dead rows are clamped to the last row and
    must not be written), with NaN guard rows around the output; B = 2 where a CTA spans both samples."""
    rpc = rows_per_cta(dim)
    rng = _rng("tail", dim)
    w16 = bf16_values(1 + 0.1 * rng.standard_normal(dim))
    for tail in range(1, rpc):
        rows = 2 * rpc + tail
        x = _rows(rng, rows, dim, 0.3)
        xt = _bf16(x)
        sc, sh = (rng.standard_normal((2, 1, dim)) * 0.5).astype(np.float32)
        cos, sin = _tables(rng, rows)
        buf, out = _fenced(rows, dim)
        _abi_ln(xt, None, None, _f32(sc), _f32(sh), out, rows)
        torch.cuda.synchronize()
        assert _guards_intact(buf, rows, dim), f"ln_modulate wrote outside its {rows} rows"
        check_bar(_np(out), ln_ref(x, None, None, sc, sh), f"ln {rows} rows")
        buf, out = _fenced(rows, dim)
        _abi_rms(xt, _bf16(w16), _f32(cos), _f32(sin), out, rows)
        torch.cuda.synchronize()
        assert _guards_intact(buf, rows, dim), f"rmsnorm_rope wrote outside its {rows} rows"
        check_bar(_np(out), rms_ref(x, w16, cos, sin), f"rms {rows} rows")
    # B = 2, S not a multiple of the rows per CTA: one CTA holds rows of both samples
    S = 3 * rpc + 1
    x = _rows(rng, 2 * S, dim)
    sc, sh = (rng.standard_normal((2, 2, dim))).astype(np.float32)
    check_bar(run_ln(x, sc=sc, sh=sh, rows_per_batch=S), ln_ref(x, None, None, sc, sh, rows_per_batch=S), "B = 2")
    cos, sin = _tables(rng, S)
    check_bar(run_rms(x, w16, cos, sin, tokens_per_batch=S), rms_ref(x, w16, cos, sin, tokens_per_batch=S), "rms B = 2")


@pytest.mark.parametrize("B,S,dim", [(1, 333, 1536), (2, 130, 5120), (2, 77, 1536), (2, 5, 640), (2, 4000, 1536)])
def test_gate_residual(B, S, dim):
    """x + y * gate; gate None; B = 2 with rows * dim / 8 not a multiple of the block (2 x 77 x 1536, 2 x 5 x 640) and
    more vectors than one grid-stride pass (2 x 4000 x 1536); cancellation x ~ -y * gate."""
    rng = _rng("gate", B, S, dim)
    x, y = _rows(rng, B * S, dim), _rows(rng, B * S, dim)
    gate = rng.standard_normal((B, dim)).astype(np.float32)
    xt, yt = _bf16(x).view(B, S, dim), _bf16(y).view(B, S, dim)
    out = _np(ops.gate_residual(xt, yt, _f32(gate)).view(B * S, dim))
    ref = gate_ref(x, y, gate, rows_per_batch=S)
    check_bar(out, ref, "gate")
    check_bias(out, ref[0], "gate")
    check_bar(_np(ops.gate_residual(xt, yt, None).view(B * S, dim)), gate_ref(x, y), "no gate")
    xc = bf16_values(-(y * np.repeat(gate, S, 0)) + rng.standard_normal(y.shape) * 2.0 ** -9)
    out = _np(ops.gate_residual(_bf16(xc).view(B, S, dim), yt, _f32(gate)).view(B * S, dim))
    check_bar(out, gate_ref(xc, y, gate, rows_per_batch=S), "x ~ -y * gate")


RMS_DISPATCH = ([(d // HEAD, False) for d in WARP_DIMS] + [(h, True) for h in (12, 24, 40)]
                + [(3, False), (5, False), (64, False)])


@pytest.mark.parametrize("heads,fallback", RMS_DISPATCH,
                         ids=[f"{h * HEAD}-{'fallback' if fb else 'dispatch'}" for h, fb in RMS_DISPATCH])
def test_rmsnorm_rope_every_dispatch(heads, fallback):
    """Wan norm_q / norm_k: RMSNorm over the whole row * weight, RoPE per head with token = row % S (B = 2); random and
    exact (0, pi/2, pi, 3pi/2) angles; heads of very different scale, so a per-head norm would show."""
    dim = heads * HEAD
    rng = _rng("rms", heads, fallback)
    B, S = 2, 11
    x = bf16_values(rng.standard_normal((B * S, dim)) * np.repeat(2.0 ** (np.arange(heads) % 4), HEAD))
    w = bf16_values(1 + 0.1 * rng.standard_normal(dim))
    for exact in (False, True):
        cos, sin = _tables(rng, S, exact)
        check_bar(run_rms(x, w, cos, sin, S, fallback), rms_ref(x, w, cos, sin, tokens_per_batch=S, fallback=fallback),
                  f"exact angles {exact}")
    if not fallback:
        check_bar(run_rms(x, w), rms_ref(x, w), "norm only")


@pytest.mark.parametrize("B,S,heads", [(1, 200, 12), (2, 77, 40), (1, 96, 3), (1, 53, 24), (1, 5, 16)])
def test_rmsnorm_rope(B, S, heads):
    dim = heads * HEAD
    rng = _rng("rms-shapes", B, S, heads)
    x = _rows(rng, B * S, dim)
    w = bf16_values(1 + 0.1 * rng.standard_normal(dim))
    cos, sin = _tables(rng, S)
    check_bar(run_rms(x, w, tokens_per_batch=S), rms_ref(x, w, tokens_per_batch=S), "norm only")
    check_bar(run_rms(x, w, cos, sin, S), rms_ref(x, w, cos, sin, tokens_per_batch=S), "rope")


def _headnorm_np(x, w, heads, cos=None, sin=None, rope_rows=None, out=None, dst_row0=0):
    xt = _bf16(x)
    got = ops.headnorm_rope(xt, None if w is None else _bf16(w), 1e-6, heads, None if cos is None else _f32(cos),
                            None if sin is None else _f32(sin), rope_rows=rope_rows, out=out, dst_row0=dst_row0)
    return got


@pytest.mark.parametrize("B,S,T,heads", [(1, 200, 16, 24), (2, 77, 9, 3), (1, 1030, 256, 24), (1, 5, 0, 16),
                                         (2, 7, 5, 3), (1, 1, 1, 1)])
def test_headnorm_rope_joint_sequence(B, S, T, heads):
    """HunyuanVideo Q / K prologue (hunyuan.py:62-134): per-head RMSNorm, RoPE on the video rows only, rows placed in the
    joint [video | text] tensor at dst_row0 = 0 and S, in a NaN-filled buffer whose other rows must stay untouched;
    the single-stream form in place with rope_rows = S; rope_rows 0 and all rows; unit counts B * rows * heads that
    are not a multiple of 4 half-warps (2 x 7 x 3, 1 x 1 x 1)."""
    dim = heads * HEAD
    rng = _rng("headnorm", B, S, T, heads)
    xv = bf16_values(rng.standard_normal((B, S, dim)) * np.repeat(2.0 ** (np.arange(heads) % 4), HEAD))
    xt = bf16_values(rng.standard_normal((B, T, dim)))
    wv, wt = (bf16_values(1 + 0.1 * rng.standard_normal(HEAD)) for _ in range(2))
    cos, sin = _tables(rng, S)
    buf, joint2 = _fenced(B * (S + T), dim)
    joint = joint2.view(B, S + T, dim)
    _headnorm_np(xv, wv, heads, cos, sin, out=joint)
    torch.cuda.synchronize()
    assert _guards_intact(buf, B * (S + T), dim), "headnorm_rope wrote outside its destination"
    assert bool((joint[:, S:].contiguous().view(torch.int16) == NAN16).all()), "video rows leaked into the text rows"
    if T:
        _headnorm_np(xt, wt, heads, out=joint, dst_row0=S)
        torch.cuda.synchronize()
        assert _guards_intact(buf, B * (S + T), dim), "headnorm_rope wrote outside its destination"
    rv, Ev = headnorm_ref(xv, wv, heads, cos, sin)
    rt, Et = headnorm_ref(xt, wt, heads)
    check_bar(_np(joint), (np.concatenate([rv, rt], 1), np.concatenate([Ev, Et], 1)), "joint")
    # single stream: one tensor over the joint sequence, in place, RoPE on the first S rows
    both = np.concatenate([xv, xt], 1)
    bt = _bf16(both)
    got = ops.headnorm_rope(bt, _bf16(wv), 1e-6, heads, _f32(cos), _f32(sin), rope_rows=S)
    assert got.data_ptr() == bt.data_ptr()
    cos_all, sin_all = _tables(rng, S + T)
    check_bar(_np(got), headnorm_ref(both, wv, heads, cos, sin, rope_rows=S), "in place, rope_rows = S")
    for rr in (0, S + T):
        got = _headnorm_np(both, wv, heads, cos_all, sin_all, rope_rows=rr)
        check_bar(_np(got), headnorm_ref(both, wv, heads, cos_all, sin_all, rope_rows=rr), f"rope_rows {rr}")
    with pytest.raises(ValueError):
        ops.headnorm_rope(_bf16(xv), _bf16(wv), 1e-6, heads, out=joint, dst_row0=T + 1)        # does not fit


@pytest.mark.parametrize("heads", [1, 3, 24])
def test_headnorm_rope_exact_angles_without_norm(heads):
    """weight=None with rotation by exact table angles: angle 0 returns x, pi/2 maps (re, im) to (-im, re), pi negates,
    bit for bit; with a norm the same tables stay within the bar."""
    rng = _rng("exact", heads)
    B, S = 2, 9
    x = _rows(rng, B * S, heads * HEAD).reshape(B, S, heads * HEAD)
    k = rng.integers(0, 4, (S, HEAD // 2))
    cos = np.choose(k, [1, 0, -1, 0]).astype(np.float32)
    sin = np.choose(k, [0, 1, 0, -1]).astype(np.float32)
    got = _np(_headnorm_np(x, None, heads, cos, sin))
    want = headnorm_ref(x, None, heads, cos, sin)[0]
    assert np.array_equal(got, want)
    zero = _np(_headnorm_np(x, None, heads, np.ones_like(cos), np.zeros_like(sin)))
    assert np.array_equal(zero, x)
    w = bf16_values(1 + 0.1 * rng.standard_normal(HEAD))
    check_bar(_np(_headnorm_np(x, w, heads, cos, sin)), headnorm_ref(x, w, heads, cos, sin), "norm + exact angles")


# ---------------------------------------------------------------------------------------------------------------------
# host checks: malformed input raises ValueError before any launch
# ---------------------------------------------------------------------------------------------------------------------
def _raises_without_launch(fn):
    torch.cuda.synchronize()
    ops.stats_reset()
    with pytest.raises(ValueError):
        fn()
    assert ops.stats()[0] == 0


def test_block_ops_reject_malformed_input_without_launching():
    B, S, dim = 2, 5, 1536
    x = torch.randn((B, S, dim), device="cuda").bfloat16()
    v = torch.randn(dim, device="cuda")
    sc = torch.randn((B, dim), device="cuda")
    # y must be bf16
    _raises_without_launch(lambda: ops.gate_residual(x, x.float(), sc))
    # weight / bias of the wrong length
    _raises_without_launch(lambda: ops.ln_modulate(x, v[:-8], None))
    _raises_without_launch(lambda: ops.ln_modulate(x, None, v[:-8]))
    # per-token or otherwise foreign modulation shapes
    for bad in (torch.randn((B, S, dim), device="cuda"), torch.randn((3, dim), device="cuda"),
                torch.randn((B, 2, dim), device="cuda"), torch.randn((dim + 8,), device="cuda")):
        _raises_without_launch(lambda: ops.ln_modulate(x, None, None, bad, bad))
        _raises_without_launch(lambda: ops.gate_residual(x, x, bad))
    _raises_without_launch(lambda: ops.ln_modulate(x, None, None, sc, None))
    # modulation on the host
    _raises_without_launch(lambda: ops.ln_modulate(x, None, None, sc.cpu(), sc.cpu()))
    # rmsnorm: weight length, sin shape / dtype
    cos = torch.rand((S, 64), device="cuda")
    w16 = torch.ones(dim, device="cuda").bfloat16()
    _raises_without_launch(lambda: ops.rmsnorm_rope(x, w16[:-128], 1e-6))
    _raises_without_launch(lambda: ops.rmsnorm_rope(x, w16, 1e-6, cos, cos[:-1]))
    _raises_without_launch(lambda: ops.rmsnorm_rope(x, w16, 1e-6, cos, cos.double()))
    _raises_without_launch(lambda: ops.rmsnorm_rope(x, w16, 1e-6, cos, None))
    _raises_without_launch(lambda: ops.headnorm_rope(x, w16[:128], 1e-6, 12, cos, cos[:-1]))
    # misaligned activations: a contiguous view that starts 8 bytes past a 16-byte boundary
    flat = torch.zeros(B * S * dim + 4, device="cuda").bfloat16()
    xm = flat[4:].view(B, S, dim)
    assert xm.is_contiguous() and xm.data_ptr() % 16 == 8
    _raises_without_launch(lambda: ops.ln_modulate(xm))
    _raises_without_launch(lambda: ops.gate_residual(x, xm))
    _raises_without_launch(lambda: ops.gate_residual(xm, x))
    _raises_without_launch(lambda: ops.rmsnorm_rope(xm, w16, 1e-6))
    _raises_without_launch(lambda: ops.headnorm_rope(xm, None, 1e-6, 12))
    _raises_without_launch(lambda: ops.headnorm_rope(x, None, 1e-6, 12, out=xm))


def test_block_ops_accept_broadcast_modulation_and_copy_misaligned_parameters():
    """(dim,), (1, dim), (B, dim) and (B, 1, dim) modulation are one thing; misaligned weights and tables are copied to
    aligned storage and give the result of aligned ones, bit for bit."""
    B, S, dim = 2, 7, 1536
    x = torch.randn((B, S, dim), device="cuda").bfloat16()
    y = torch.randn((B, S, dim), device="cuda").bfloat16()
    one = torch.randn(dim, device="cuda")
    full = one.expand(B, dim).contiguous()
    want = ops.ln_modulate(x, None, None, full, -full)
    gwant = ops.gate_residual(x, y, full)
    for form in (one, one[None], one[None, None], full[:, None]):
        assert torch.equal(ops.ln_modulate(x, None, None, form, -form), want)
        assert torch.equal(ops.gate_residual(x, y, form), gwant)
    sc = torch.randn((B, dim), device="cuda")
    assert torch.equal(ops.ln_modulate(x, _misaligned(one.cpu().numpy()), None, _misaligned(sc.cpu().numpy()),
                                       _misaligned(sc.cpu().numpy())), ops.ln_modulate(x, one, None, sc, sc))
    w16 = torch.randn(dim + 1, device="cuda").bfloat16()
    wm = w16[1:]
    assert wm.data_ptr() % 16 == 2
    cos, sin = torch.rand((S, 64), device="cuda"), torch.rand((S, 64), device="cuda")
    cm, sm = _misaligned(cos.cpu().numpy()), _misaligned(sin.cpu().numpy())
    assert torch.equal(ops.rmsnorm_rope(x, wm, 1e-6, cm, sm), ops.rmsnorm_rope(x, wm.clone(), 1e-6, cos, sin))
    assert torch.equal(ops.headnorm_rope(x.clone(), wm[:128], 1e-6, 12, cm, sm),
                       ops.headnorm_rope(x.clone(), wm[:128].clone(), 1e-6, 12, cos, sin))


def test_hunyuan_fused_prologue_equals_eager_steps():
    """The processors' fused q / k / v path against the reference-shaped eager steps (same module, same inputs)."""
    from oracle import fixtures as FX
    from vorta_b200.attention import HunyuanVideoFlashAttnProcessor
    S, T, H = 128, 16, 3
    proc = HunyuanVideoFlashAttnProcessor()
    c, s = FX.hunyuan_rotary(S, 14)
    rope = (c.cuda(), s.cuda())
    for dual in (True, False):
        attn = FX.FakeHunyuanAttn(H, dual=dual, seed=11).to("cuda", torch.bfloat16)
        assert proc._qkv_fused(attn, FX.det_tensor((1, S, H * 128), 12).to("cuda", torch.bfloat16),
                               FX.det_tensor((1, T, H * 128), 13).to("cuda", torch.bfloat16), rope) is None   # grad mode
        hs = FX.det_tensor((1, S, H * 128), 12).to("cuda", torch.bfloat16)
        ehs = FX.det_tensor((1, T, H * 128), 13).to("cuda", torch.bfloat16)
        with torch.no_grad():
            fused = proc._qkv_fused(attn, hs, ehs, rope)
            q, k, v = proc._step_to_qkv_and_unflatten(attn, hs, ehs)
            q, k = proc._step_qk_norm(attn, q, k)
            q, k = proc._step_rotary_emb(attn, q, k, T, rope)
            eager = proc._step_encoder_to_qkv_and_concat(attn, q, k, v, ehs)
        assert fused is not None
        for a, b in zip(fused, eager):
            assert a.shape == b.shape
            scale = b.float().abs().max().item()
            assert (a.float() - b.float()).abs().max().item() <= 2.0 ** -6 * scale      # two bf16 roundings apart
        assert torch.equal(fused[2], eager[2])                                           # V: same GEMM, no arithmetic after
