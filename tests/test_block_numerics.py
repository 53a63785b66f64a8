"""The fp64 bar of the DiT block's fused elementwise kernels (vb_block.cu), and the proof on the CPU that it is sharp.

Every output element is compared with the same operation in fp64, computed from the bf16 inputs and the fp32 (or bf16)
parameters exactly as the kernel receives them.  The allowed error is

    |out - ref| <= ulp_bf16(ref) / 2 + 2 E

where E bounds the error of the kernel's fp32 value before its one bf16 rounding (cvt.rn).  The factor 2: with c the
bf16 value nearest to ref and t the kernel's fp32 value, |bf16(t) - t| <= |c - t| <= |c - ref| + E.  E is derived from
the kernel's operation order, with u = 2^-24 (fp32 unit roundoff), gamma(k) = k u / (1 - k u), and always from the
magnitudes of the terms, never of the result (so shift ~ -t (1 + scale) or x ~ -y gate gets no unfairly tight bound):

* Sums.  A sum whose terms each pass through at most K fp32 additions is within gamma(K) sum |terms|.  The warp-per-row
  kernels (NV = dim / 256 vectors, WPR = 1, 2 or 4 warps per row, NVT = NV / WPR vectors per thread) add NVT * 8 values
  per thread, then 5 shuffle levels, then WPR partials: K = 8 NVT + 5 + WPR.  The CTA-per-row fallback adds up to
  8 ceil(dim / 2048) values per thread, 5 shuffle levels and 3 across its 8 warps: K = 8 ceil(dim / 2048) + 8.
  headnorm adds 8 values per lane and 4 half-warp shuffle levels: K = 12.  The scaling by 1 / dim (a rounded fp32
  constant times the sum, or a division) adds 2 to K.
* LayerNorm.  The mean is off by D <= gamma(K + 2) sum |x| / n.  Each d = fl(x - mean) is off by (1 + u) D + u |d|; as
  sum (x - mu) = 0 the variance of the rounded d is (var + D^2)(1 + theta), |theta| <= gamma(K + 4) (the square's two
  roundings, the fma chain, the scaling).  Adding eps rounds once; rsqrtf is documented at 2 ulp (<= 4 u relative).
  With V = var + eps, r = V^-1/2, phi = (D^2 + gamma(K + 4)(var + D^2) + u V) / V the relative error of rstd is
  rho = phi (1 + phi) / 2 + 4 u, and t = fl(d rstd) is within  E_t = r D (1 + rho + u) + |t| (2 u + rho)(1 + rho).
* Affine t w + b (fma or two roundings): E = |w| E_t + 2 u ((|t| + E_t) |w| + |b|); bias alone: E_t + u (|t| + E_t + |b|).
* adaLN y (1 + scale) + shift: 1 + scale rounds once, then fma or two roundings:
  E = |a| E_y + u (|y| + E_y) |a| + 2 u ((|y| + E_y) |a| (1 + u) + |shift|),  a = 1 + scale.
* RMSNorm.  The mean square is within gamma(K + 2) of itself (squares of bf16 values are exact in the fma), + eps rounds
  once, rsqrtf 4 u: rho = (gamma(K + 2) + u) / 2 + 4 u; x rinv w rounds twice: E_y = |y| (rho + 2 u)(1 + rho).
  headnorm with no weight does not normalise: E_y = 0.
* RoPE re c - im s (and re s + im c), c, s the fp32 table entries: E = |c| E_re + |s| E_im + 2 u ((|re| + E_re)|c| +
  (|im| + E_im)|s|).
* Gated residual fma(y, gate, x): E = u (|x| + |y gate|); the plain add: u (|x| + |y|).

For a well-conditioned row, 2 E is a small fraction of half an ulp (test_bar_is_tight_for_well_conditioned_rows), so the
bar demands the correctly rounded result except within a few fp32 ulps of a rounding midpoint; where the fp64 result is
a bf16 value and 2 E is below a quarter ulp, the output must equal it bit for bit (checked directly by the GPU tests:
constant rows give bf16(shift), exact RoPE angles without a norm permute and negate x).

The bar is proven sharp here, without a GPU: numpy fp32 emulators of each kernel (the loop order of every thread, the
shuffle trees, the dead-row clamp, the pair index of the RoPE, fma where the kernel writes fmaf) pass it on every probe,
and each injected fault fails on the probe built for it:
F1 the one-pass variance sum(x^2)/n - mean^2 (rows with |mean| / std ~ 200); F2 eps dropped or doubled (variance ~ eps);
F3 bf16 rounding by truncation (mean signed relative error); F4 scale / shift of the CTA's first row's sample (B = 2 with
S not a multiple of the rows per CTA); F5 the RoPE pair index from tid & 31, and sin with the wrong sign; F6 a per-head
norm where the whole row is normalised (Wan norm_q / norm_k) and the reverse (HunyuanVideo normalises each head).
"""
import math

import numpy as np
import pytest
import torch

F32 = np.float32
U = 2.0 ** -24                   # fp32 unit roundoff
HEAD = 128
BIAS_MAX = 2.0 ** -12            # mean signed relative error of the elements with |ref| >= 2^-4


def gamma(k):
    return k * U / (1 - k * U)


# ---------------------------------------------------------------------------------------------------------------------
# dispatch geometry (vb_block.cu: row_warps, launch_ln_modulate / launch_rmsnorm_rope)
# ---------------------------------------------------------------------------------------------------------------------
WARP_DIMS = tuple(nv * 256 for nv in (4, 6, 8, 12, 16, 20, 24))


def row_warps(nv):
    return 4 if nv > 12 else 2 if nv > 6 else 1


def rows_per_cta(dim):
    return 256 // (32 * row_warps(dim // 256))


def sum_depth(dim, fallback):
    """K of the row sums of the kernel that runs at this width."""
    if fallback or dim not in WARP_DIMS:
        return 8 * (-(-dim // 2048)) + 8
    nv = dim // 256
    wpr = row_warps(nv)
    return 8 * (nv // wpr) + 5 + wpr


# ---------------------------------------------------------------------------------------------------------------------
# fp64 references with their fp32 error bound E
# ---------------------------------------------------------------------------------------------------------------------
def _per_row(p, rows, rows_per_batch, dim):
    """(batch, dim) per-sample parameter -> (rows, dim) as the kernels index it (batch = row / rows_per_batch)."""
    p = np.asarray(p, np.float64).reshape(-1, dim)
    return p[np.arange(rows) // rows_per_batch]


def ln_ref(x, w=None, b=None, scale=None, shift=None, eps=1e-6, rows_per_batch=None, fallback=False):
    """x (rows, dim) of bf16 values; w, b (dim,); scale, shift (batch, dim).  Returns (ref, E)."""
    x = np.asarray(x, np.float64)
    rows, n = x.shape
    rows_per_batch = rows if rows_per_batch is None else rows_per_batch
    K = sum_depth(n, fallback)
    mu = x.mean(1, keepdims=True)
    d = x - mu
    var = (d * d).mean(1, keepdims=True)
    V = var + eps
    r = 1.0 / np.sqrt(V)
    t = d * r
    D = gamma(K + 2) * np.abs(x).sum(1, keepdims=True) / n
    phi = (D * D + gamma(K + 4) * (var + D * D) + U * V) / V
    rho = phi * (1 + phi) / 2 + 4 * U
    E = r * D * (1 + rho + U) + np.abs(t) * (2 * U + rho) * (1 + rho)
    y = t
    if w is not None:
        w = np.asarray(w, np.float64)
        bb = np.zeros(n) if b is None else np.asarray(b, np.float64)
        E = np.abs(w) * E + 2 * U * ((np.abs(y) + E) * np.abs(w) + np.abs(bb))
        y = y * w + bb
    elif b is not None:
        bb = np.asarray(b, np.float64)
        E = E + U * (np.abs(y) + E + np.abs(bb))
        y = y + bb
    if scale is not None:
        a = 1 + _per_row(scale, rows, rows_per_batch, n)
        sh = _per_row(shift, rows, rows_per_batch, n)
        E = np.abs(a) * E + U * (np.abs(y) + E) * np.abs(a) + 2 * U * ((np.abs(y) + E) * np.abs(a) * (1 + U) + np.abs(sh))
        y = y * a + sh
    return y, E


def _rope(y, E, cos, sin, tok):
    """Rotate channel pairs (2i, 2i+1) of every 128-wide head of y (rows, dim) by cos / sin [tok[row], i]."""
    rows, n = y.shape
    c = np.tile(np.asarray(cos, np.float64)[tok], (1, n // HEAD))
    s = np.tile(np.asarray(sin, np.float64)[tok], (1, n // HEAD))
    re, im, Er, Ei = y[:, 0::2], y[:, 1::2], E[:, 0::2], E[:, 1::2]
    out, Eo = np.empty_like(y), np.empty_like(E)
    mag = 2 * U * ((np.abs(re) + Er) * np.abs(c) + (np.abs(im) + Ei) * np.abs(s))
    out[:, 0::2] = re * c - im * s
    out[:, 1::2] = re * s + im * c
    Eo[:, 0::2] = np.abs(c) * Er + np.abs(s) * Ei + mag
    Eo[:, 1::2] = np.abs(s) * Er + np.abs(c) * Ei + mag
    return out, Eo


def rms_ref(x, w, cos=None, sin=None, eps=1e-6, tokens_per_batch=None, fallback=False):
    """Wan norm_q / norm_k + RoPE: RMSNorm over the whole row * w (bf16 values), token = row % tokens_per_batch."""
    x = np.asarray(x, np.float64)
    rows, n = x.shape
    K = sum_depth(n, fallback)
    R = 1.0 / np.sqrt((x * x).mean(1, keepdims=True) + eps)
    rho = (gamma(K + 2) + U) / 2 + 4 * U
    y = x * R * np.asarray(w, np.float64)
    E = np.abs(y) * (rho + 2 * U) * (1 + rho)
    if cos is not None:
        tpb = rows if tokens_per_batch is None else tokens_per_batch
        y, E = _rope(y, E, cos, sin, np.arange(rows) % tpb)
    return y, E


def headnorm_ref(x, w, heads, cos=None, sin=None, eps=1e-6, rope_rows=None):
    """HunyuanVideo: x (B, rows, heads*128); per-head RMSNorm * w (128) (None: no norm), RoPE on rows < rope_rows."""
    x = np.asarray(x, np.float64)
    B, rows, n = x.shape
    xh = x.reshape(B, rows, heads, HEAD)
    if w is not None:
        R = 1.0 / np.sqrt((xh * xh).mean(-1, keepdims=True) + eps)
        rho = (gamma(12 + 2) + U) / 2 + 4 * U
        yh = xh * R * np.asarray(w, np.float64)
        Eh = np.abs(yh) * (rho + 2 * U) * (1 + rho)
    else:
        yh, Eh = xh.copy(), np.zeros_like(xh)
    y, E = yh.reshape(B * rows, n), Eh.reshape(B * rows, n)
    if cos is not None:
        nr = rows if rope_rows is None else rope_rows
        r_idx = np.tile(np.arange(rows), B)
        sel = r_idx < nr
        if sel.any():
            y[sel], E[sel] = _rope(y[sel], E[sel], cos, sin, r_idx[sel])
    return y.reshape(B, rows, n), E.reshape(B, rows, n)


def gate_ref(x, y, gate=None, rows_per_batch=None):
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    rows, n = x.shape
    if gate is None:
        return x + y, U * (np.abs(x) + np.abs(y))
    g = _per_row(gate, rows, rows if rows_per_batch is None else rows_per_batch, n)
    return x + y * g, U * (np.abs(x) + np.abs(y * g))


# ---------------------------------------------------------------------------------------------------------------------
# the bar
# ---------------------------------------------------------------------------------------------------------------------
def half_ulp(ref):
    a = np.abs(np.asarray(ref, np.float64))
    e = np.floor(np.log2(np.maximum(a, 2.0 ** -126)))
    return 2.0 ** (e - 8)


def bar_excess(out, ref, E):
    """(|out - ref| - tol) / half_ulp(ref) per element: > 0 where the bar fails (NaN counts as a failure)."""
    out = np.asarray(out, np.float64)
    err = np.abs(out - ref)
    ex = (err - (half_ulp(ref) + 2 * E)) / half_ulp(ref)
    return np.where(np.isnan(ex), np.inf, ex)


def check_bar(out, ref_E, what=""):
    """out within the bar of ref_E = (ref, E)."""
    ref, E = ref_E
    ex = bar_excess(out, ref, E)
    bad = ex > 0
    if bad.any():
        i = np.unravel_index(int(np.argmax(ex)), ex.shape)
        out = np.asarray(out, np.float64)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} elements outside the bar; worst at {i}: out "
                             f"{out[i]!r}, ref {ref[i]!r}, E {E[i]:.3g}, half ulp {half_ulp(ref)[i]:.3g}")


def signed_bias(out, ref):
    """Mean of sign(ref) (out - ref) / |ref| over the elements with |ref| >= 2^-4: round to nearest leaves ~0."""
    out = np.asarray(out, np.float64)
    m = np.abs(ref) >= 2.0 ** -4
    return float(np.mean(np.sign(ref[m]) * (out[m] - ref[m]) / np.abs(ref[m])))


def check_bias(out, ref, what=""):
    b = signed_bias(out, ref)
    assert abs(b) <= BIAS_MAX, f"{what}: mean signed relative error {b:.3g} (bf16 rounding not to nearest?)"


# ---------------------------------------------------------------------------------------------------------------------
# fp32 emulators of the kernels (vectorised over rows; each loop follows one thread's order)
# ---------------------------------------------------------------------------------------------------------------------
def bf16_round(a):
    return torch.from_numpy(np.ascontiguousarray(a, F32)).bfloat16().float().numpy().astype(np.float64)


def bf16_trunc(a):
    bits = np.ascontiguousarray(a, F32).view(np.uint32) & np.uint32(0xFFFF0000)
    return bits.view(F32).astype(np.float64)


def fma32(a, b, c):
    return (np.float64(1) * a * b + c).astype(F32)


def rsqrt32(v):
    return (1.0 / np.sqrt(np.asarray(v, np.float64))).astype(F32)


def _butterfly(a, levels):
    """xor-shuffle sum over the last axis (lanes), levels = (16, 8, ...)."""
    lanes = np.arange(a.shape[-1])
    for o in levels:
        a = (a + a[..., lanes ^ o]).astype(F32)
    return a


def _warp_row_sum(parts, wpr):
    """parts (rows, 32 * wpr) per-thread fp32 partials -> row_sum<WPR>: warp butterfly, then warps 0..WPR-1 from 0."""
    a = _butterfly(parts.reshape(parts.shape[0], wpr, 32), (16, 8, 4, 2, 1))[:, :, 0]
    if wpr == 1:
        return a[:, 0]
    r = np.zeros(a.shape[0], F32)
    for i in range(wpr):
        r = (r + a[:, i]).astype(F32)
    return r


def _block_sum(parts):
    """parts (rows, 256) -> block_sum2: butterfly per warp, lane 0 of warp w to red[w], butterfly 4, 2, 1 over red."""
    a = _butterfly(parts.reshape(parts.shape[0], 8, 32), (16, 8, 4, 2, 1))[:, :, 0]
    return _butterfly(a, (4, 2, 1))[:, 0]


def _warp_layout(x, dim):
    """(rows, NVT, 32 * WPR, 8): vector idx = i * 32 * WPR + tid of the warp-per-row kernels."""
    wpr = row_warps(dim // 256)
    return x.reshape(x.shape[0], dim // 256 // wpr, 32 * wpr, 8), wpr


def _cta_layout(x, dim):
    """(rows, kMaxVec, 256, 8) with zero padding past nvec: vector idx = threadIdx.x + i * 256 of the fallback."""
    nvec = dim // 8
    nslots = -(-nvec // 256)
    pad = np.zeros((x.shape[0], nslots * 256 * 8), F32)
    pad[:, :dim] = x
    return pad.reshape(x.shape[0], nslots, 256, 8), nvec


def _thread_sums(lay, valid, f):
    """Sequential per-thread sum over (i, e) of f(value); lay (rows, I, T, 8); valid (I, T) bool."""
    s = np.zeros(lay.shape[0:1] + lay.shape[2:3], F32)
    for i in range(lay.shape[1]):
        for e in range(8):
            s = np.where(valid[i], f(lay[:, i, :, e], s), s).astype(F32)
    return s


def emulate_ln(x, w=None, b=None, scale=None, shift=None, eps=1e-6, rows_per_batch=None, fallback=False, fault=None):
    """vb_ln_modulate_warp_kernel<NV> or vb_ln_modulate_kernel on x (rows, dim) bf16 values.  Faults: "one_pass",
    "no_eps", "double_eps", "truncate", "cta_batch"."""
    x = np.asarray(x, F32)
    rows, dim = x.shape
    rows_per_batch = rows if rows_per_batch is None else rows_per_batch
    eps32 = F32(eps) * (0 if fault == "no_eps" else 2 if fault == "double_eps" else 1)
    add = lambda v, s: (s + v).astype(F32)
    sq = lambda v, s: fma32(v, v, s)
    if fallback or dim not in WARP_DIMS:
        lay, nvec = _cta_layout(x, dim)
        valid = (np.arange(lay.shape[1])[:, None] * 256 + np.arange(256)[None]) < nvec
        mean = (_block_sum(_thread_sums(lay, valid, add)).astype(np.float64) / dim).astype(F32)[:, None]
        if fault == "one_pass":
            ms = (_block_sum(_thread_sums(lay, valid, sq)).astype(np.float64) / dim).astype(F32)[:, None]
            var = np.maximum(fma32(-mean, mean, ms), F32(0))
        else:
            dl = (lay - mean[:, :, None, None]).astype(F32)
            var = (_block_sum(_thread_sums(dl, valid, sq)).astype(np.float64) / dim).astype(F32)[:, None]
        rstd = rsqrt32((var + eps32).astype(F32))
    else:
        lay, wpr = _warp_layout(x, dim)
        valid = np.ones(lay.shape[1:3], bool)
        inv = F32(1.0 / dim)
        mean = (_warp_row_sum(_thread_sums(lay, valid, add), wpr) * inv).astype(F32)[:, None]
        if fault == "one_pass":
            ms = (_warp_row_sum(_thread_sums(lay, valid, sq), wpr) * inv).astype(F32)[:, None]
            var = np.maximum(fma32(-mean, mean, ms), F32(0))
        else:
            dl = (lay - mean[:, :, None, None]).astype(F32)
            var = (_warp_row_sum(_thread_sums(dl, valid, sq), wpr) * inv).astype(F32)[:, None]
        rstd = rsqrt32((var + eps32).astype(F32))
    t = ((x - mean).astype(F32) * rstd).astype(F32)
    if w is not None:
        t = fma32(t, np.asarray(w, F32), F32(0) if b is None else np.asarray(b, F32))
    elif b is not None:
        t = (t + np.asarray(b, F32)).astype(F32)
    if scale is not None:
        row = np.arange(rows)
        if fault == "cta_batch":
            rpc = rows_per_cta(dim)
            row = row // rpc * rpc
        sc = np.asarray(scale, F32).reshape(-1, dim)[row // rows_per_batch]
        sh = np.asarray(shift, F32).reshape(-1, dim)[row // rows_per_batch]
        t = fma32(t, (F32(1) + sc).astype(F32), sh)
    return bf16_trunc(t) if fault == "truncate" else bf16_round(t)


def _rope32(y, cos, sin, tok, pair, fault):
    """y (rows, dim) fp32; pair (dim / 2,) pair index of every channel pair inside the table row."""
    ct = np.concatenate([np.asarray(cos, F32).reshape(-1), np.zeros(HEAD, F32)])   # a read past a row takes the
    st = np.concatenate([np.asarray(sin, F32).reshape(-1), np.zeros(HEAD, F32)])   # next token's entries
    idx = tok[:, None] * (HEAD // 2) + pair[None]
    c, s = ct[idx], st[idx]
    if fault == "sin_sign":
        s = -s
    re, im = y[:, 0::2], y[:, 1::2]
    out = np.empty_like(y)
    out[:, 0::2] = fma32(re, c, -(im * s).astype(F32))
    out[:, 1::2] = fma32(re, s, (im * c).astype(F32))
    return out


def emulate_rms(x, w, cos=None, sin=None, eps=1e-6, tokens_per_batch=None, fallback=False, fault=None):
    """vb_rmsnorm_rope_warp_kernel<NV> or vb_rmsnorm_rope_kernel.  Faults: "pair_tid31", "sin_sign", "per_head"."""
    x = np.asarray(x, F32)
    rows, dim = x.shape
    sq = lambda v, s: fma32(v, v, s)
    if fault == "per_head":
        h = x.reshape(rows, dim // HEAD, HEAD).astype(np.float64)
        ms = (h * h).mean(2).astype(F32)
        rinv = np.repeat(rsqrt32((ms + F32(eps)).astype(F32)), HEAD, axis=1)
    elif fallback or dim not in WARP_DIMS:
        lay, nvec = _cta_layout(x, dim)
        valid = (np.arange(lay.shape[1])[:, None] * 256 + np.arange(256)[None]) < nvec
        ms = (_block_sum(_thread_sums(lay, valid, sq)).astype(np.float64) / dim).astype(F32)
        rinv = rsqrt32((ms + F32(eps)).astype(F32))[:, None]
    else:
        lay, wpr = _warp_layout(x, dim)
        ss = _warp_row_sum(_thread_sums(lay, np.ones(lay.shape[1:3], bool), sq), wpr)
        rinv = rsqrt32(fma32(ss, F32(1.0 / dim), F32(eps)))[:, None]
    y = ((x * rinv).astype(F32) * np.asarray(w, F32)).astype(F32)
    if cos is not None:
        tpb = rows if tokens_per_batch is None else tokens_per_batch
        pair = (np.arange(dim // 2) % (HEAD // 2))
        if fault == "pair_tid31" and not (fallback or dim not in WARP_DIMS):
            # the warp kernel's thread tid owns channel pairs 4 tid .. 4 tid + 3 of its vectors; & 31 instead of & 15
            tid = (np.arange(dim // 8) % (32 * row_warps(dim // 256)))
            pair = np.repeat((tid & 31) * 4, 4) + np.tile(np.arange(4), dim // 8)
        y = _rope32(y, cos, sin, np.arange(rows) % tpb, pair, fault)
    return bf16_round(y)


def emulate_headnorm(x, w, heads, cos=None, sin=None, eps=1e-6, rope_rows=None, fault=None):
    """vb_headnorm_rope_kernel on x (B, rows, heads*128): half-warp per (row, head), 8 fma per lane, butterfly 8..1.
    Faults: "whole_row" (one norm over all heads of a row), "sin_sign"."""
    x = np.asarray(x, F32)
    B, rows, dim = x.shape
    units = x.reshape(B * rows * heads, 16, 8)
    y = units.copy()
    if w is not None:
        if fault == "whole_row":
            rr = x.reshape(B * rows, dim).astype(np.float64)
            ms = np.repeat(((rr * rr).mean(1)).astype(F32), heads)
            rinv = rsqrt32((ms + F32(eps)).astype(F32))
        else:
            s = np.zeros((units.shape[0], 16), F32)
            for e in range(8):
                s = fma32(units[:, :, e], units[:, :, e], s)
            s = _butterfly(s, (8, 4, 2, 1))[:, 0]
            rinv = rsqrt32(fma32(s, F32(1.0 / HEAD), F32(eps)))
        y = ((units * rinv[:, None, None]).astype(F32) * np.asarray(w, F32).reshape(16, 8)).astype(F32)
    y = y.reshape(B * rows, dim)
    if cos is not None:
        nr = rows if rope_rows is None else rope_rows
        r_idx = np.tile(np.arange(rows), B)
        sel = r_idx < nr
        y[sel] = _rope32(y[sel], cos, sin, r_idx[sel], np.arange(dim // 2) % (HEAD // 2), fault)
    return bf16_round(y).reshape(B, rows, dim)


# ---------------------------------------------------------------------------------------------------------------------
# probes
# ---------------------------------------------------------------------------------------------------------------------
def bf16_values(a):
    return bf16_round(np.asarray(a, np.float64))


def ln_rows(rng, rows, dim, offset=0.0, std=1.0):
    """bf16 rows N(offset, std^2)."""
    return bf16_values(rng.standard_normal((rows, dim)) * std + offset)


def mod_params(rng, batch, dim, s=0.2):
    return (rng.standard_normal((batch, dim)) * s).astype(F32), (rng.standard_normal((batch, dim)) * s).astype(F32)


def rope_tables(rng, tokens):
    ang = rng.random((tokens, HEAD // 2)) * 2 * math.pi
    return np.cos(ang).astype(F32), np.sin(ang).astype(F32)


def excess(emulated, ref_E):
    return float(bar_excess(emulated, *ref_E).max())


LN_CASES = [(dim, fb) for dim in WARP_DIMS for fb in (False, True)] + [(384, True), (640, True), (8192, True)]


@pytest.mark.parametrize("dim,fallback", LN_CASES)
def test_faithful_ln_emulator_passes_every_probe(dim, fallback):
    rng = np.random.default_rng(dim + fallback)
    rows = 12
    for offset in (0.0, 0.3, 16.0, 64.0, 200.0):
        x = ln_rows(rng, rows, dim, offset)
        check_bar(emulate_ln(x, fallback=fallback), ln_ref(x, fallback=fallback), f"offset {offset}")
    x = ln_rows(rng, rows, dim, 0.0, 1e-3)                                                      # variance ~ eps
    check_bar(emulate_ln(x, fallback=fallback), ln_ref(x, fallback=fallback), "var ~ eps")
    x = ln_rows(rng, rows, dim, 0.0, 1e4)
    check_bar(emulate_ln(x, fallback=fallback), ln_ref(x, fallback=fallback), "1e4")
    x = np.repeat(bf16_values(rng.standard_normal((rows, 1))), dim, 1)                          # constant rows
    sc, sh = mod_params(rng, 2, dim)
    sh = bf16_values(np.sign(sh) * (0.5 + 10 * np.abs(sh))).astype(F32)                      # |shift| >= 1/2
    kw = dict(scale=sc, shift=sh, rows_per_batch=rows // 2 + 1, fallback=fallback)
    out = emulate_ln(x, **kw)
    check_bar(out, ln_ref(x, **kw), "constant rows")
    assert np.array_equal(out, _per_row(sh, rows, rows // 2 + 1, dim)), "constant row -> bf16(shift)"
    w = (1 + 0.1 * rng.standard_normal(dim)).astype(F32)
    b = (0.1 * rng.standard_normal(dim)).astype(F32)
    x = ln_rows(rng, rows, dim, 0.5, 2.0)
    for kw in (dict(w=w, b=b, scale=sc, shift=sh), dict(b=b), dict(w=w)):
        kw.update(rows_per_batch=rows // 2, fallback=fallback)
        check_bar(emulate_ln(x, **kw), ln_ref(x, **kw), str(sorted(kw)))
    # cancellation: shift ~ -t (1 + scale)
    t, _ = ln_ref(x[:2])
    sc1 = sc[:1]
    sh1 = (-(t[:1] * (1 + sc1)) + rng.standard_normal((1, dim)) * 1e-3).astype(F32)
    kw = dict(scale=sc1, shift=sh1, fallback=fallback)
    check_bar(emulate_ln(x[:1], **kw), ln_ref(x[:1], **kw), "shift ~ -t (1 + scale)")


@pytest.mark.parametrize("dim", [1536, 3072, 5120, 8192, 640])
def test_f1_one_pass_variance_fails_at_mean_over_std_200(dim):
    rng = np.random.default_rng(1)
    x = ln_rows(rng, 16, dim, 200.0)
    fb = dim not in WARP_DIMS or dim == 5120
    ref = ln_ref(x, fallback=fb)
    assert excess(emulate_ln(x, fallback=fb), ref) <= 0
    assert excess(emulate_ln(x, fallback=fb, fault="one_pass"), ref) > 0


@pytest.mark.parametrize("dim,fallback", [(1536, False), (4096, False), (384, True), (3072, True)])
@pytest.mark.parametrize("fault", ["no_eps", "double_eps"])
def test_f2_eps_dropped_or_doubled_fails_at_variance_near_eps(dim, fallback, fault):
    rng = np.random.default_rng(2)
    x = ln_rows(rng, 8, dim, 0.0, 1e-3)
    ref = ln_ref(x, fallback=fallback)
    assert excess(emulate_ln(x, fallback=fallback), ref) <= 0
    assert excess(emulate_ln(x, fallback=fallback, fault=fault), ref) > 0
    ref = rms_ref(x, np.ones(dim), fallback=fallback)
    assert excess(emulate_rms(x, np.ones(dim), fallback=fallback), ref) <= 0


@pytest.mark.parametrize("dim,fallback", [(2048, False), (640, True)])
def test_f3_truncation_fails_the_mean_signed_error(dim, fallback):
    rng = np.random.default_rng(3)
    x = ln_rows(rng, 64, dim, 0.3, 2.0)
    ref, _ = ln_ref(x, fallback=fallback)
    check_bias(emulate_ln(x, fallback=fallback), ref)
    with pytest.raises(AssertionError):
        check_bias(emulate_ln(x, fallback=fallback, fault="truncate"), ref)


@pytest.mark.parametrize("dim", [1536, 3072, 6144])
def test_f4_modulation_of_the_wrong_sample_fails_when_a_cta_spans_two_samples(dim):
    rng = np.random.default_rng(4)
    rpc = rows_per_cta(dim)
    S = 3 * rpc + 1 if rpc > 1 else 3                  # S not a multiple of rows per CTA (2 rows per CTA: S odd)
    x = ln_rows(rng, 2 * S, dim)
    sc, sh = mod_params(rng, 2, dim, 1.0)
    kw = dict(scale=sc, shift=sh, rows_per_batch=S)
    ref = ln_ref(x, **kw)
    assert excess(emulate_ln(x, **kw), ref) <= 0
    assert excess(emulate_ln(x, **kw, fault="cta_batch"), ref) > 0


@pytest.mark.parametrize("dim,fallback", [(1024, False), (3072, False), (5120, False), (1536, True), (384, True)])
def test_faithful_rms_emulator_and_f5_rope_faults(dim, fallback):
    rng = np.random.default_rng(5 + dim)
    B, S = 2, 7
    x = ln_rows(rng, B * S, dim)
    w = bf16_values(1 + 0.1 * rng.standard_normal(dim))
    cos, sin = rope_tables(rng, S)
    kw = dict(cos=cos, sin=sin, tokens_per_batch=S, fallback=fallback)
    ref = rms_ref(x, w, **kw)
    assert excess(emulate_rms(x, w, **kw), ref) <= 0
    check_bar(emulate_rms(x, w, fallback=fallback), rms_ref(x, w, fallback=fallback), "norm only")
    assert excess(emulate_rms(x, w, **kw, fault="sin_sign"), ref) > 0
    if not fallback:
        assert excess(emulate_rms(x, w, **kw, fault="pair_tid31"), ref) > 0


@pytest.mark.parametrize("dim", [1536, 5120, 384])
def test_f6_per_head_norm_in_place_of_the_whole_row_fails(dim):
    rng = np.random.default_rng(6)
    heads = dim // HEAD
    x = bf16_values(rng.standard_normal((6, dim)) * np.repeat(2.0 ** (np.arange(heads) % 4), HEAD))
    w = bf16_values(1 + 0.1 * rng.standard_normal(dim))
    ref = rms_ref(x, w)
    assert excess(emulate_rms(x, w), ref) <= 0
    assert excess(emulate_rms(x, w, fault="per_head"), ref) > 0


@pytest.mark.parametrize("B,rows,heads,rope_rows", [(1, 9, 3, 9), (2, 5, 24, 3), (2, 4, 2, 0)])
def test_faithful_headnorm_emulator_and_f5_f6_faults(B, rows, heads, rope_rows):
    rng = np.random.default_rng(7 + heads)
    x = bf16_values(rng.standard_normal((B, rows, heads * HEAD)) * np.repeat(2.0 ** (np.arange(heads) % 4), HEAD))
    w = bf16_values(1 + 0.1 * rng.standard_normal(HEAD))
    cos, sin = rope_tables(rng, rows)
    kw = dict(cos=cos, sin=sin, rope_rows=rope_rows)
    ref = headnorm_ref(x, w, heads, **kw)
    assert excess(emulate_headnorm(x, w, heads, **kw), ref) <= 0
    assert excess(emulate_headnorm(x, None, heads, **kw), headnorm_ref(x, None, heads, **kw)) <= 0
    assert excess(emulate_headnorm(x, w, heads, **kw, fault="whole_row"), ref) > 0
    if rope_rows:
        assert excess(emulate_headnorm(x, w, heads, **kw, fault="sin_sign"), ref) > 0


def test_bar_is_tight_for_well_conditioned_rows():
    """2 E stays a small fraction of half an ulp: the bar demands the correctly rounded result almost everywhere."""
    rng = np.random.default_rng(8)
    for dim, fb in ((1536, False), (6144, False), (8192, True)):
        x = ln_rows(rng, 4, dim, 0.3)
        sc, sh = mod_params(rng, 1, dim)
        for ref, E in (ln_ref(x, fallback=fb), ln_ref(x, scale=sc, shift=sh, fallback=fb),
                       rms_ref(x, bf16_values(np.ones(dim)), *rope_tables(rng, 4), fallback=fb)):
            m = np.abs(ref) >= 2.0 ** -4
            assert float((2 * E[m] / half_ulp(ref[m])).max()) < 0.125
    x, y = ln_rows(rng, 4, 1536), ln_rows(rng, 4, 1536)
    ref, E = gate_ref(x, y, rng.standard_normal((1, 1536)))
    m = np.abs(ref) >= 2.0 ** -4
    assert float((2 * E[m] / half_ulp(ref[m])).max()) < 0.125


def test_bar_rejects_one_ulp_everywhere():
    rng = np.random.default_rng(9)
    x = ln_rows(rng, 8, 2048, 0.3)
    ref, E = ln_ref(x)
    out = emulate_ln(x)
    check_bar(out, (ref, E))
    nudged = bf16_values(out * (1 + 2.0 ** -7))                 # one ulp up (about) everywhere
    assert float((bar_excess(nudged, ref, E) > 0).mean()) > 0.5
