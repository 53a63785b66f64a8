"""The softmax weights of the attention kernel against fp64: read-out probes of single weights, the lazy rescale and the
row maximum at their edges, keys that are loaded but must not be attended, and peaked logits at full size.

test_gpu_attn_exact.py pins which keys each row attends to and where each row lands, with inputs whose softmax is
either flat or one-hot; test_gpu_parity.py compares randn inputs with a cosine / max-abs bar, under which a 5 % error on
the polynomial exponential lanes or a truncated P still passes.  Here every output element is held to a bound derived
from the kernel's arithmetic (vb_attn.cu, softmax warps; vb_ptx.cuh, exp2_poly2):

* x_j = s_j * scale_log2 - m_ref in fp32 (one FMA), m_ref the row maximum of the first block, raised only when a later
  block's maximum exceeds it by more than 2^8 (kRescaleThreshold, log2 units); O and l are then both scaled by
  ex2(m_ref - m_new), which cancels in O / l.
* e_j = 2^x_j: keys 4-7 of every 32 columns of a block through exp2_poly2 (relative error below EPS_EXP), the rest
  through ex2.approx.ftz (PTX ISA: 2 ulp, far below EPS_EXP).
* P_j = bf16(e_j), round to nearest (relative error <= U = 2^-8); l = sum of the unrounded e_j in fp32.
* O = sum P_j v_j accumulated by the tensor core in fp32; the output is bf16(O / l).

Write w_j = 2^(x_j - m) with the exact logits x_j = (q . k_j) * log2(e) / sqrt(128) and the exact maximum m, p_j = w_j /
sum w, O* = sum p_j v_j.  The kernel's exponential of key j is w_j (1 + a_j) up to a factor common to the row, with
|a_j| <= (1 + EPS_EXP) 2^dx_j - 1, where dx_j bounds the error of the kernel's logit in log2 units:

    dx_j = scale_log2 * C_QK * sum_i |q_i k_ji|  +  2^-22 (|x_j - m| + 1)

C_QK = 2^-14 covers the fp32 tensor-core accumulation of the 128 exact bf16 products (its rounding is not IEEE and not
documented; 2^-14 is four times the 2^-16 of 128 truncated fp32 additions), the second term the fp32 constant
scale_log2 and the fp32 FMA.  With P_j = e_j (1 + r_j), |r_j| <= U, and abar = sum p_j |a_j|:

    |O~ - O*| <= [sum_j p_j (|a_j| + U + U |a_j|) |v_j| + abar |O*|] / (1 - abar)

to which are added the fp32 accumulation of O and l (EPS_ACC per 16-key MMA step, per rescale and per partial sum of l,
times sum p_j |v_j|), the output rounding U |O*|, and an absolute 2^-125 per key whose exponential underflows (x_j - m
< -100: ex2.approx.ftz flushes, bf16 subnormals may be flushed by the tensor core).  Where no attended key has a
non-zero value in a channel the reference is exactly 0, and so must the output be.  Blend mode: sum_e w_e bound_e plus
one output rounding.

The bar is proven sharp without a GPU: a CPU emulator of the kernel's softmax (128-key blocks along the kernel's run
lists, the lane pattern, exp2_poly2 bit for bit, bf16 P, fp32 l, the lazy rescale, the tail mask, the max exchange of
the two half-row threads) passes it on every probe input, and each injected fault fails it on the probes built for it:
F1 polynomial lanes 1 % off; F2 P truncated to bf16 (seen by the bias check: the mean signed relative error of the
read-out elements); F3 l, or O, not rescaled; F4 a rescale threshold of 128; F5 the row maximum taken before the tail
mask; F6 each half-row thread using its own half's maximum; F7 a masked key with a non-zero weight (exp2_poly2 once
clamped -inf to 2^-126).
"""
import math

import numpy as np
import pytest
import torch

from oracle import vorta_oracle as O
from vorta_b200 import _lib as L
from vorta_b200 import ops

from test_gpu_attn_exact import HUNYUAN, TEXT, WAN13, WAN14, to_dev, window_keys

gpu = pytest.mark.gpu

U = 2.0 ** -8                    # bf16 unit roundoff (P and the output)
EPS_EXP = 7.6e-5                 # exp2_poly2's relative error: 7.497e-5 of the polynomial plus its fp32 roundings (the
                                 # emulation below: 7.503e-5); ex2.approx.ftz is 2 ulp
C_QK = 2.0 ** -14                # tensor-core fp32 accumulation of QK, relative to sum |q_i k_i|
EPS_STEP = 2.0 ** -22            # one fp32 accumulation step of O or l, relative to the magnitudes summed so far
SCALE_LOG2 = math.log2(math.e) / math.sqrt(128)
SCALE_F32 = np.float32(np.float32(1.4426950408889634) / np.sqrt(np.float32(128)))   # the kernel's p.scale_log2
BIAS_MAX = 3 * 2.0 ** -12        # mean signed relative error of the read-out elements
THRESHOLD = 8.0                  # kRescaleThreshold
POISON_NATS = 300.0              # logit of a key that is loaded but not attended, above every attended key
POISON_CODE = 2.0 ** 20          # its value, in a channel no attended key uses


class Group:
    """Query rows that share one run list: q (R, 128), k / v (n, 128) in kernel order (rows past n read as 0, as TMA
    fills them), runs [(start, len)] in the order the kernel walks them, rows: where the R rows sit in the output."""

    def __init__(self, q, k, v, runs, rows, name):
        self.q, self.k, self.v, self.rows, self.name = q, k, v, rows, name
        self.runs = [(int(s), int(n)) for s, n in runs]

    def keys(self):
        return torch.cat([torch.arange(s, s + n) for s, n in self.runs])

    def n_blocks(self):
        return sum(-(-n // 128) for _, n in self.runs)


# ---------------------------------------------------------------------------------------------------------
# the bar
# ---------------------------------------------------------------------------------------------------------
def reference(g):
    """(O*, bound, zero) float64 (R, 128): the fp64 softmax output over the group's keys, the allowed error of each
    element (module docstring) and where the output must be exactly 0."""
    keys = g.keys()
    K, V = g.k[keys].double(), g.v[keys].double()
    q = g.q.double()
    x = (q @ K.T) * SCALE_LOG2
    d = x - x.max(dim=1, keepdim=True).values
    w = torch.exp2(d)
    p = w / w.sum(dim=1, keepdim=True)
    want = p @ V
    dx = SCALE_LOG2 * C_QK * (q.abs() @ K.abs().T) + 2.0 ** -22 * (d.abs() + 1)
    a = (1 + EPS_EXP) * torch.exp2(dx) - 1
    tiny = d < -100
    a = torch.where(tiny, torch.ones_like(a), a)
    abar = (p * a).sum(dim=1, keepdim=True)
    assert float(abar.max()) < 0.25, "the probe's logits are too large for a first-order bound"
    T = p @ V.abs()
    Ta = (p * (a + U + U * a)) @ V.abs()
    nu = 2.0 ** -125 * (tiny.double() @ V.abs())
    eps_acc = EPS_STEP * (len(keys) / 16 + 3 * g.n_blocks() + 24)
    bound = (Ta + abar * want.abs()) / (1 - abar) + eps_acc * (1 + U) * (1 + abar) / (1 - abar) * T + nu
    bound = U * want.abs() + (1 + U) * bound + 2.0 ** -120
    zero = (V.abs().sum(dim=0) == 0).expand_as(want)
    return want, bound, zero


def failures(got, want, bound, zero):
    got = got.double()
    err = (got - want).abs()
    return ~torch.isfinite(got) | (zero & (got != 0)) | (~zero & ~(err <= bound))


def ratio(got, want, bound, zero):
    err = ((got.double() - want).abs() / bound)[~zero]
    return float(err.max()) if err.numel() else 0.0


def assert_within_bound(got, want, bound, zero, what=""):
    bad = failures(got, want, bound, zero)
    if bad.any():
        i = tuple(int(x) for x in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside the bound, first at {i}: got "
                             f"{float(got.double()[i])}, want {float(want[i])}, bound {float(bound[i])}, "
                             f"zero {bool(zero[i])}")
    return ratio(got, want, bound, zero)


def bias(got, want, zero):
    sel = ~zero & (want.abs() > 2.0 ** -100)
    return float(((got.double() - want) / want.abs())[sel].mean())


# ---------------------------------------------------------------------------------------------------------
# the emulator
# ---------------------------------------------------------------------------------------------------------
_M = np.float32(12582912.0)
_C = [np.float32(c) for c in (0.055171020, 0.24260981, 0.69326097, 0.99992818)]


def _fma(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def exp2_poly2(x, clamp_to_constant=False):
    """exp2_poly2 bit for bit: clamp at -126, x = n + f by the 1.5 * 2^23 trick, Horner in fp32 FMA, n added to the
    exponent field as an integer.  Below -126 the kernel returns exactly 0 (clamp_to_constant: the old 2^-126 * p(0))."""
    x = np.asarray(x, dtype=np.float32)
    xc = np.maximum(x, np.float32(-126.0))
    t = (xc + _M).astype(np.float32)
    r = (t - _M).astype(np.float32)
    f = _fma(r, np.float32(-1.0), xc)
    p = _fma(f, _C[0], _C[1])
    p = _fma(p, f, _C[2])
    p = _fma(p, f, _C[3])
    e = (p.view(np.uint32) + (t.view(np.uint32) << np.uint32(23))).view(np.float32)
    return e if clamp_to_constant else np.where(x < -126, np.float32(0), e)


def ex2_ftz(x):
    e = np.exp2(np.asarray(x, dtype=np.float64)).astype(np.float32)
    return np.where(e < np.float32(2.0 ** -126), np.float32(0), e)


def to_bf16(x, truncate=False):
    x = np.ascontiguousarray(x, dtype=np.float32)
    if truncate:
        return (x.view(np.uint32) & np.uint32(0xFFFF0000)).view(np.float32)
    return torch.from_numpy(x).to(torch.bfloat16).float().numpy()


COL = np.arange(128)
POLY = (COL % 32 >= 4) & (COL % 32 < 8)          # kPolyGroups = 0x02
HALF = COL // 64


def emulate(g, fault=None):
    """The kernel's softmax and PV over the group's run list, (R, 128) float64 of the bf16 output."""
    q = g.q.double().numpy()
    k, v = g.k.double().numpy(), g.v.double().numpy()
    n, R = k.shape[0], q.shape[0]
    thr = np.float32(128.0 if fault == "F4" else THRESHOLD)
    m_ref = np.zeros((R, 2), np.float32)            # per half-row thread; equal in both unless F6
    l = np.zeros((R, 2), np.float32)
    acc = np.zeros((R, 128), np.float64)
    first = True
    for start, length in g.runs:
        for off in range(0, length, 128):
            valid = min(128, length - off)
            idx = start + off + COL
            inside = idx < n
            kb, vb = np.zeros((128, 128)), np.zeros((128, 128))
            kb[inside], vb[inside] = k[idx[inside]], v[idx[inside]]
            s = (q @ kb.T).astype(np.float32)
            masked = np.where(COL >= valid, np.float32(-np.inf), s)
            src = s if fault == "F5" else masked
            mh = np.stack([src[:, :64].max(axis=1), src[:, 64:].max(axis=1)], axis=1)
            if fault != "F6":
                mh = np.repeat(mh.max(axis=1, keepdims=True), 2, axis=1)
            m_new = (mh * SCALE_F32).astype(np.float32)
            if first:
                m_ref = m_new
            else:
                need = m_new > m_ref + thr
                alpha = np.where(need, ex2_ftz(m_ref.astype(np.float64) - m_new), np.float32(1))
                m_ref = np.where(need, m_new, m_ref)
                if fault != "F3o":
                    acc *= np.repeat(alpha, 64, axis=1)
                if fault != "F3l":
                    l = (l * alpha).astype(np.float32)
            x = (masked.astype(np.float64) * np.float64(SCALE_F32) - m_ref[:, HALF]).astype(np.float32)
            e = np.where(POLY, exp2_poly2(x, clamp_to_constant=fault == "F7"), ex2_ftz(x))
            if fault == "F1":
                e = np.where(POLY, (e * np.float32(1.01)).astype(np.float32), e)
            for h in range(2):
                l[:, h] = (l[:, h] + e[:, 64 * h:64 * h + 64].astype(np.float64).sum(axis=1)).astype(np.float32)
            P = to_bf16(e, truncate=fault == "F2")
            kst = -(-valid // 16) * 16                 # PV covers the valid keys rounded up to 16
            acc += P[:, :kst].astype(np.float64) @ vb[:kst]
            first = False
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        out = (acc.astype(np.float32) / (l[:, 0] + l[:, 1])[:, None]).astype(np.float32)
    return torch.from_numpy(to_bf16(out)).double()


# ---------------------------------------------------------------------------------------------------------
# 3. read-out probes: K = one-hot of the column, V = one-hot of the column, so output channel c is the weight of the
# key in column c of the last block
# ---------------------------------------------------------------------------------------------------------
def bf(x):
    return torch.as_tensor(x, dtype=torch.float64).to(torch.bfloat16).double()


def readout_sweep(R=512):
    """Two blocks.  Block 0: 128 keys with logit A_r (K = e_127, V = 0) fix m_ref = A_r * scale; block 1: key c has K =
    e_c and V = e_c, so x_c = (Q[r, c] - A_r) * scale.  Targets cover [-140, 7] on every lane (below the rescale
    threshold); A_r in steps of 1/16 moves every row's fractional parts through a whole unit, so f passes +-0.5."""
    r = torch.arange(R)
    A = bf((r % 128).double() / 16)
    c = torch.arange(127)
    target = -140.0 + ((r[:, None] * 7 + c[None] * 13) % 147).double() + 0.5
    q = torch.zeros((R, 128), dtype=torch.float64)
    q[:, :127] = bf(target / SCALE_LOG2 + A[:, None])
    q[:, 127] = A
    k = torch.zeros((256, 128), dtype=torch.float64)
    v = torch.zeros_like(k)
    k[:128, 127] = 1.0
    k[128:] = torch.eye(128, dtype=torch.float64)
    v[128:] = torch.eye(128, dtype=torch.float64)
    return Group(q, k, v, [(0, 256)], None, "read-out sweep")


def readout_tail(n_k, R=300, extra=8):
    """One block of n_k keys (K = e_c, V = e_c), the row maximum A_r on key r mod n_k, the rest [-140, 0] below it.
    K and V are prefixes of allocations with `extra` poison rows: logit 300 nats above the maximum (channel 127), value
    POISON_CODE in channel 127 (n_k = 128: K 0, POISON_CODE in every channel)."""
    r = torch.arange(R)
    A = bf((r % 128).double() / 16)
    c = torch.arange(n_k)
    target = -140.0 + ((r[:, None] * 11 + c[None] * 29) % 140).double()
    target[r, r % n_k] = 0.0
    q = torch.zeros((R, 128), dtype=torch.float64)
    q[:, :n_k] = bf(target / SCALE_LOG2 + A[:, None])
    q[r, r % n_k] = A
    k = torch.zeros((n_k + extra, 128), dtype=torch.float64)
    v = torch.zeros_like(k)
    k[:n_k, :n_k] = torch.eye(n_k, dtype=torch.float64)
    v[:n_k, :n_k] = torch.eye(n_k, dtype=torch.float64)
    if n_k < 128:
        q[:, 127] = 1.0
        k[n_k:, 127] = float(bf((POISON_NATS + 20) * math.sqrt(128)))
        v[n_k:, 127] = POISON_CODE
    else:
        v[n_k:] = POISON_CODE
    return Group(q, k[:n_k], v[:n_k], [(0, n_k)], None, f"read-out tail {n_k}"), k, v


TAILS = (1, 5, 17, 100, 128)


def readout_cases():
    return [readout_sweep()] + [readout_tail(n)[0] for n in TAILS]


# ---------------------------------------------------------------------------------------------------------
# 4. lazy-rescale edges: a "boost" key per slot (its own channel 120 + i) raises a row's maximum by a chosen growth
# ---------------------------------------------------------------------------------------------------------
DELTA = 0.25
GROWTHS = (0.0, THRESHOLD - DELTA, THRESHOLD + DELTA, 127.0, 140.0)


def base_qkv(N, seed, B=1, H=1):
    """Channels [0, 120) randn * 0.5 (logit std ~0.25 nats: no rescale of its own), V randn; float64 bf16 values."""
    g = torch.Generator().manual_seed(seed)
    q = torch.zeros((B, H, N, 128), dtype=torch.float64)
    k = torch.zeros_like(q)
    q[..., :120] = bf(0.5 * torch.randn((B, H, N, 120), generator=g, dtype=torch.float64))
    k[..., :120] = bf(0.5 * torch.randn((B, H, N, 120), generator=g, dtype=torch.float64))
    v = bf(torch.randn((B, H, N, 128), generator=g, dtype=torch.float64))
    return q, k, v, g


def plant_growth(q, k, v, rows, order, runs, slots, channel0, g):
    """Rows `rows` (raster) attend the kernel-order keys of `runs`; kernel position i -> raster order[i].  Slot j is
    the kernel-order key slots[j]: it gets K = 1 in channel channel0 + j and V = +-4 (so that a growth of 127 left
    unrescaled overflows fp32), and row r the growth GROWTHS[...] above its first block's maximum on slot r mod len."""
    first = torch.arange(runs[0][0], runs[0][0] + min(128, runs[0][1]))
    for j, pos in enumerate(slots):
        key = int(order[pos])
        k[key, channel0 + j] = 1.0
        v[key] = 4.0 * torch.where(torch.rand(128, generator=g) < 0.5, -1.0, 1.0).double()
    for i, row in enumerate(rows.tolist()):
        j = i % len(slots)
        growth = GROWTHS[(i // len(slots) + i) % len(GROWTHS)]
        if growth == 0:
            continue
        m0 = float((k[order[first]] @ q[row]).max()) * SCALE_LOG2
        key = int(order[slots[j]])
        base = float(k[key, :120] @ q[row, :120])
        q[row, channel0 + j] = float(bf((m0 + growth) / SCALE_LOG2 - base))
        real = (float(k[key] @ q[row]) * SCALE_LOG2) - m0
        assert abs(real - growth) < (0.1 if growth < 100 else 0.7), (growth, real)


DENSE_SLOTS = [128 + 5, 128 + 70, 128 + 10, 128 + 90, 384 + 37, 384 + 100, 640 + 4, 640 + 1]   # block 1, 3, tail


def rescale_dense(n_q=256, n_k=645):
    """Blocks 0-4 full and a 5-key tail block: growth at block 1, a middle block and the tail, on polynomial and MUFU
    lanes, in both halves, with rows of one warp deciding differently."""
    q, k, v, g = base_qkv(max(n_q, n_k), 5)
    q, k, v = q[0, 0, :n_q].clone(), k[0, 0, :n_k].clone(), v[0, 0, :n_k].clone()
    plant_growth(q, k, v, torch.arange(n_q), torch.arange(n_k), [(0, n_k)], DENSE_SLOTS, 120, g)
    return Group(q, k, v, [(0, n_k)], torch.arange(n_q), "rescale dense")


def sliding_schedule(plan):
    """[(raster query tokens, runs, split tile)] of every query tile of the sliding branch, from the plan's export."""
    runs = plan.export(L.EXPORT_SLIDING_RUNS).reshape(-1, 2)
    items = plan.export(L.EXPORT_SLIDING_ITEMS).reshape(-1, 12)
    qmap = torch.from_numpy(plan.export(L.EXPORT_SLIDING_QUERY_MAP).astype(np.int64))
    out = []
    for it in items.tolist():
        for t in range(it[6]):
            second = bool(it[8]) and t == 1
            rb, rc = (it[9], it[10]) if second else (it[4], it[5])
            out.append((qmap[it[t]:it[t] + it[2 + t]], runs[rb:rb + rc].tolist(), second))
    return out


def kernel_order(plan, branch):
    """Kernel-order key position -> raster token (full: raster itself; sliding: tile-major video, then text)."""
    S, N = plan.seq_len, plan.seq_len + plan.text_len
    if branch == 0:
        return torch.arange(N)
    return torch.cat([O.tile_permutation(plan.latent_shape, plan.tile_size), torch.arange(S, N)])


def tiles_of(plan, tokens):
    inv = torch.argsort(O.tile_permutation(plan.latent_shape, plan.tile_size))
    return set((inv[tokens[tokens < plan.seq_len]] // plan.tile_tokens).tolist())


def sliding_group_of_tile(plan, tile, split=False):
    """The schedule entry (query tokens, runs) holding query tile `tile`; its key set is checked against the oracle."""
    for rows, runs, second in sliding_schedule(plan):
        if second == split and tile in tiles_of(plan, rows):
            pos, _ = window_keys(plan.latent_shape, plan.tile_size, plan.window_size, tile)
            S = plan.seq_len
            got = torch.cat([torch.arange(s, s + n) for s, n in runs])
            want = torch.cat([pos, torch.arange(S, S + plan.text_valid)])
            assert torch.equal(got.sort().values, want), f"tile {tile}: run list != oracle window"
            return rows, runs
    raise AssertionError(f"no {'split ' if split else ''}query tile {tile}")


def routed_group(plan, q, k, v, branch, rows, runs, name):
    """The kernel's tensor maps end at S + text_valid: padded text keys are read as zeros."""
    order = kernel_order(plan, branch)[:plan.seq_len + plan.text_valid]
    return Group(q[rows], k[order], v[order], runs, rows, name)


SPLIT = ((6, 6, 8), (1, 3, 4), (3, 3, 3), (2, 3, 2), 0, 0)


def rescale_routed():
    """[(geometry, branch, q, k, v, groups)]: full head with text (growth in blocks 1, 2, the tail and the text keys);
    Wan-14B sliding (first block of a second run, the 16-key tail of a 1296-key run); HunyuanVideo sliding (growth in
    the text run only); a split work item's second tile."""
    out = []
    lat, tile, win, lw, tl, tv = TEXT
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    S = plan.seq_len
    q, k, v, g = base_qkv(S + tl, 41)
    q, k, v = q[0, 0], k[0, 0], v[0, 0]
    rows, runs = torch.arange(S + tv), [(0, S + tv)]
    plant_growth(q, k, v, rows, kernel_order(plan, 0), runs, [128 + 5, 128 + 74, 256 + 36, 512 + 4, 512 + 50,
                                                              S + 4, S + 10], 120, g)
    out.append((TEXT, 0, q, k, v, [routed_group(plan, q, k, v, 0, rows, runs, "rescale full+text")]))

    for geom, tiles, name in ((WAN14, (87, 0), "wan14"), (HUNYUAN, (131,), "hunyuan text run")):
        lat, tile, win, lw, tl, tv = geom
        plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
        S = plan.seq_len
        q, k, v, g = base_qkv(S + tl, 43)
        q, k, v = q[0, 0], k[0, 0], v[0, 0]
        groups = []
        for i, t in enumerate(tiles):
            rows, runs = sliding_group_of_tile(plan, t)
            if tv:
                assert runs[-1] == [S, tv]
                slots = [S + 4, S + 40]
            else:
                assert runs[0][1] == 1296 and len(runs) >= 2
                slots = [runs[1][0] + 5, runs[1][0] + 66, runs[0][0] + 1280 + 4, runs[0][0] + 1280 + 9]
            plant_growth(q, k, v, rows, kernel_order(plan, 2), runs, slots, 120 + 4 * i, g)
            groups.append(routed_group(plan, q, k, v, 2, rows, runs, f"rescale {name} tile {t}"))
        out.append((geom, 2, q, k, v, groups))

    lat, tile, win, lw, tl, tv = SPLIT
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    items = plan.export(L.EXPORT_SLIDING_ITEMS).reshape(-1, 12)
    assert int(items[:, 8].sum()) >= 1, "the geometry has no split item"
    q, k, v, g = base_qkv(plan.seq_len, 47)
    q, k, v = q[0, 0], k[0, 0], v[0, 0]
    rows, runs, _ = next(e for e in sliding_schedule(plan) if e[2])
    assert sum(n for _, n in runs) > 128
    first_len = runs[0][1]
    blk1 = runs[0][0] + 128 if first_len > 128 else runs[1][0]
    plant_growth(q, k, v, rows, kernel_order(plan, 2), runs, [blk1 + 5, blk1 + 9], 120, g)
    out.append((SPLIT, 2, q, k, v, [routed_group(plan, q, k, v, 2, rows, runs, "rescale split item")]))
    return out


# ---------------------------------------------------------------------------------------------------------
# 5. poison keys: loaded by the kernel, not attended
# ---------------------------------------------------------------------------------------------------------
# 45-token tiles: 135-key runs (tail block of 7 keys: masked columns 7-15 hold the next tile, column 7 a polynomial
# lane); the window leaves tiles out along W and T.  37 valid text keys of 48 and S + TV = 1477 put masked polynomial
# lanes behind the text run and the last full-branch block too, but there the padded text keys lie past the end of the
# kernel's tensor maps and are read as zeros: those cases check the output only
POISON = ((4, 10, 36), (1, 5, 9), (3, 3, 3), (2, 2, 2), 48, 37)


def poison_routed():
    """[(branch, tile or None / "text", q, k, v, group)]: every key a row may not attend has logit 300 nats above its attended keys (channel
    127, Q = 1) and value POISON_CODE in channel 127, which no attended key uses."""
    lat, tile, win, lw, tl, tv = POISON
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    S = plan.seq_len
    out = []
    cases = [(0, None)] + [(2, t) for t in (0, 5, 13)] + [(2, "text")]
    for branch, t in cases:
        q, k, v, _ = base_qkv(S + tl, 53 + len(out))
        q, k, v = q[0, 0], k[0, 0], v[0, 0]
        v[:, 127] = 0.0
        if t is None or t == "text":
            rows, runs = torch.arange(S, S + tv) if t else torch.arange(S + tv), [(0, S + tv)]
            if t:
                rows, runs = next((r, rr) for r, rr, _ in sliding_schedule(plan) if int(r[0]) >= S)
            attended = torch.arange(S + tv)
        else:
            rows, runs = sliding_group_of_tile(plan, t)
            order = kernel_order(plan, 2)
            attended = order[torch.cat([torch.arange(s, s + n) for s, n in runs])]
        poison = torch.ones(S + tl, dtype=torch.bool)
        poison[attended] = False
        assert poison.any()
        q[rows, 127] = 1.0
        k[poison, 127] = float(bf((POISON_NATS + 20) * math.sqrt(128)))
        v[poison, 127] = POISON_CODE
        name = f"poison {'full' if branch == 0 else 'sliding'} {t if t is not None else ''}".strip()
        out.append((branch, t, q, k, v, routed_group(plan, q, k, v, branch, rows, runs, name)))
    return plan, out


# ---------------------------------------------------------------------------------------------------------
# CPU self-checks
# ---------------------------------------------------------------------------------------------------------
def emulated_failures(g, fault):
    want, bound, zero = reference(g)
    got = emulate(g, fault)
    return bool(failures(got, want, bound, zero).any()), bias(got, want, zero)


def test_exp2_poly2_emulation():
    """The emulated exp2_poly2: relative error below EPS_EXP on [-125, 8]; exactly 0 below -126 and at -inf; the old
    clamp gave 2^-126 * p(0) there."""
    x = np.linspace(-125, 8, 400001).astype(np.float32)
    e = exp2_poly2(x).astype(np.float64)
    rel = e / np.exp2(x.astype(np.float64)) - 1
    assert np.abs(rel).max() < EPS_EXP
    assert exp2_poly2(np.float32(-np.inf)) == 0 and exp2_poly2(np.float32(-126.5)) == 0
    old = float(exp2_poly2(np.float32(-np.inf), clamp_to_constant=True))
    assert abs(old - 1.1753e-38) < 1e-42 and old < 2.0 ** -126


def test_read_out_bar_is_sharp():
    """Faithful emulator within the bound and unbiased on every read-out probe; F1 outside the bound on each of them
    that has a polynomial lane (5 keys or more), F2 biased on each of those (one key alone has weight exactly 1)."""
    for g in readout_cases():
        bad, b = emulated_failures(g, None)
        assert not bad, g.name
        assert abs(b) < BIAS_MAX / 4, (g.name, b)
        if len(g.keys()) > 4:
            assert emulated_failures(g, "F1")[0], f"{g.name}: F1 passes"
            assert emulated_failures(g, "F2")[1] < -BIAS_MAX, f"{g.name}: F2 passes the bias check"
    g = readout_sweep()
    x = (g.q[:, :127] - g.q[:, 127:]) * SCALE_LOG2
    f = x - x.round()
    poly = torch.from_numpy(POLY[:127])
    assert float(x.min()) < -139 and 6 < float(x.max()) < THRESHOLD
    assert float(f[:, poly].abs().max()) > 0.49 and float(f[:, poly].min()) < -0.49 and float(f[:, poly].max()) > 0.49


def test_rescale_bar_is_sharp():
    groups = [rescale_dense()] + [grp for *_, gs in rescale_routed() for grp in gs]
    for g in groups:
        assert not emulated_failures(g, None)[0], g.name
        for fault in ("F3l", "F3o", "F4", "F6"):
            assert emulated_failures(g, fault)[0], f"{g.name}: {fault} passes"


def test_poison_bar_is_sharp():
    """Faithful emulator within the bound on every poison probe; F5 and F7 outside it on each sliding tile, whose run
    tails are followed by poisoned keys of the neighbouring tile.  (The dense poison rows past n_k and the padded text
    keys lie past the kernel's tensor maps, which read as zeros.)"""
    _, cases = poison_routed()
    for branch, tile, *_, g in cases:
        assert not emulated_failures(g, None)[0], g.name
        if isinstance(tile, int):
            for fault in ("F5", "F7"):
                assert emulated_failures(g, fault)[0], f"{g.name}: {fault} passes"


def test_split_geometry_has_split_items():
    plan = ops.Plan(*SPLIT[:4], 0.5)
    assert int(plan.export(L.EXPORT_SLIDING_ITEMS).reshape(-1, 12)[:, 8].sum()) >= 1


# ---------------------------------------------------------------------------------------------------------
# GPU probes
# ---------------------------------------------------------------------------------------------------------
def report(name, r, extra=""):
    print(f"NUMERICS {name}: max error / bound {r:.3f} {extra}")


@gpu
def test_read_out_probes():
    g = readout_sweep()
    out = ops.attn_dense(to_dev(g.q[None, None]), to_dev(g.k[None, None]), to_dev(g.v[None, None]))[0, 0].cpu()
    want, bound, zero = reference(g)
    r = assert_within_bound(out, want, bound, zero, g.name)
    b = bias(out, want, zero)
    report(g.name, r, f"bias {b:.2e}")
    assert abs(b) < BIAS_MAX, b
    for n_k in TAILS:
        g, k_alloc, v_alloc = readout_tail(n_k)
        kd, vd = to_dev(k_alloc[None, None]), to_dev(v_alloc[None, None])
        out = ops.attn_dense(to_dev(g.q[None, None]), kd[:, :, :n_k], vd[:, :, :n_k])[0, 0].cpu()
        want, bound, zero = reference(g)
        r = assert_within_bound(out, want, bound, zero, g.name)
        b = bias(out, want, zero)
        report(g.name, r, f"bias {b:.2e}")
        assert abs(b) < BIAS_MAX, (n_k, b)


def _run_routed(geom, branch, q, k, v):
    lat, tile, win, lw, tl, tv = geom
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    flags = L.ATTN_CORESET_KV_FROM_K if tl else 0
    return ops.routed_attention(plan, to_dev(q[None, None]), to_dev(k[None, None]), to_dev(v[None, None]),
                                branch=[branch], flags=flags)[0, 0].cpu()


@gpu
def test_lazy_rescale_edges():
    g = rescale_dense()
    out = ops.attn_dense(to_dev(g.q[None, None]), to_dev(g.k[None, None]), to_dev(g.v[None, None]))[0, 0].cpu()
    report(g.name, assert_within_bound(out, *reference(g), g.name))
    for geom, branch, q, k, v, groups in rescale_routed():
        out = _run_routed(geom, branch, q, k, v)
        for g in groups:
            report(g.name, assert_within_bound(out[g.rows], *reference(g), g.name))


@gpu
def test_poison_keys_get_no_weight():
    _, cases = poison_routed()
    for branch, _, q, k, v, g in cases:
        out = _run_routed(POISON, branch, q, k, v)
        want, bound, zero = reference(g)
        got = out[g.rows]
        leak = float(got[:, 127].abs().max())
        assert zero[:, 127].all()
        report(g.name, ratio(got, want, bound, zero), f"poison channel max |O| {leak:.3e}")
        assert_within_bound(got, want, bound, zero, g.name)


# ---------------------------------------------------------------------------------------------------------
# 6. peaked parity at full size
# ---------------------------------------------------------------------------------------------------------
# Logit std in nats.  No checkpoint is available to measure the range real models reach; randn Q and K give ~1 nat,
# 12 makes most rows nearly one-hot.
LOGIT_STD = (1.0, 4.0, 12.0)


def peaked_qkv(B, H, N, std, seed):
    g = torch.Generator().manual_seed(seed)
    s = std ** 0.5
    q, k = (bf(s * torch.randn((B, H, N, 128), generator=g, dtype=torch.float64)) for _ in range(2))
    return q, k, bf(torch.randn((B, H, N, 128), generator=g, dtype=torch.float64))


def kept_tokens(q, k, info):
    """Raster ids of the coreset's kept query tokens and kept key tokens (K's own matching when k is given, as
    HunyuanVideo pools K and V; otherwise Q's), from the fp64 oracle."""
    def kept(x):
        m = O.match(x.double(), info)
        return torch.cat([info.center_indices[:, 0], O.kept_token_ids(info, m[0])[0, 0]])
    kq = kept(q)
    return kq, kept(k) if k is not None else kq


def _check_rows(out, q, k, v, rows, keys, name, blocks=None):
    """out rows `rows` against attention of q[rows] over k[keys], v[keys]."""
    g = Group(q[rows], k[keys], v[keys], [(0, len(keys))] if blocks is None else blocks, rows, name)
    r = assert_within_bound(out[rows], *reference(g), name)
    return r


def _peaked(geom, std, B=1, text_valid=None, seed=0):
    lat, tile, win, lw, tl, tv = geom
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    S, H = plan.seq_len, 3
    q, k, v = peaked_qkv(B, H, S + tl, std, seed)
    flags = L.ATTN_CORESET_KV_FROM_K if tl else 0
    qd, kd, vd = to_dev(q, "token"), to_dev(k, "token"), to_dev(v, "token")
    out = ops.routed_attention(plan, qd, kd, vd, branch=[0, 1, 2], flags=flags, text_valid=text_valid).cpu()
    info = O.get_group_info(lat, lw, 0.5)
    tvs = text_valid if text_valid is not None else [tv] * B
    worst = 0.0
    perm = O.tile_permutation(lat, tile).reshape(-1, plan.tile_tokens)
    n_tiles = perm.shape[0]
    for b in range(B):
        tvb = tvs[b]
        nv = S + tvb
        text = torch.arange(S, nv)
        o = out[b]
        tag = f"{lat} std {std} b {b}"
        # full head: sampled video rows and every valid text row
        rows = torch.cat([torch.arange(0, S, max(1, S // 48)), text])
        worst = max(worst, _check_rows(o[0], q[b, 0], k[b, 0], v[b, 0], rows, torch.arange(nv), f"full {tag}"))
        # sliding head: corner, edge and interior tiles, and the valid text rows
        for t in (0, n_tiles // 7, n_tiles // 2, n_tiles - 1):
            pos, _ = window_keys(lat, tile, win, t)
            keys = torch.cat([perm.reshape(-1)[pos], text])
            worst = max(worst, _check_rows(o[2], q[b, 2], k[b, 2], v[b, 2], perm[t], keys, f"sliding {tag} tile {t}"))
        if tvb:
            worst = max(worst, _check_rows(o[2], q[b, 2], k[b, 2], v[b, 2], text, torch.arange(nv), f"text {tag}"))
        # coreset head: sampled kept query rows (each its own pooled row) over the kept keys and the valid text
        kept_q, kept_k = kept_tokens(q[b:b + 1, 1:2], k[b:b + 1, 1:2] if tl else None, info)
        rows = kept_q[::max(1, len(kept_q) // 48)]
        worst = max(worst, _check_rows(o[1], q[b, 1], k[b, 1], v[b, 1], rows, torch.cat([kept_k, text]),
                                       f"coreset {tag}"))
    return worst


@gpu
@pytest.mark.parametrize("std", LOGIT_STD)
@pytest.mark.parametrize("geom", [WAN13, WAN14, HUNYUAN], ids=["wan13", "wan14", "hunyuan"])
def test_peaked_parity_full_size(geom, std):
    report(f"peaked {geom[0]} std {std}", _peaked(geom, std, seed=int(std)))


@gpu
def test_peaked_parity_batch2_per_sample_text():
    report("peaked hunyuan batch 2", _peaked(HUNYUAN, 4.0, B=2, text_valid=[64, 17], seed=3))


@gpu
@pytest.mark.parametrize("std", LOGIT_STD)
def test_peaked_blend_small_geometry(std):
    lat, tile, win, lw, tl, tv = TEXT
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    S, H = plan.seq_len, 3
    q, k, v = peaked_qkv(1, H, S + tl, std, 7)
    w = torch.softmax(torch.randn((1, H, 3), generator=torch.Generator().manual_seed(7)), -1)
    qd, kd, vd = to_dev(q), to_dev(k), to_dev(v)
    out = ops.routed_attention(plan, qd, kd, vd, weights=w, flags=L.ATTN_CORESET_KV_FROM_K).cpu()[0]
    info = O.get_group_info(lat, lw, 0.5)
    nv = S + tv
    perm = O.tile_permutation(lat, tile)
    text = torch.arange(S, nv)
    worst = 0.0
    for h in range(H):
        # rows: the coreset's kept query tokens (each is its own pooled row) and the valid text rows
        kept_q, kept_k = kept_tokens(q[:, h:h + 1], k[:, h:h + 1], info)
        rows = torch.cat([kept_q.sort().values, text])
        ref = []
        full = reference(Group(q[0, h, rows], k[0, h, :nv], v[0, h, :nv], [(0, nv)], rows, "full"))
        ref.append(full[:2])
        keys = torch.cat([kept_k, text])
        ref.append(reference(Group(q[0, h, rows], k[0, h, keys], v[0, h, keys], [(0, len(keys))], rows, "cs"))[:2])
        want_s = torch.zeros((len(rows), 128), dtype=torch.float64)
        bound_s = torch.zeros_like(want_s)
        where = {int(r): i for i, r in enumerate(rows.tolist())}
        inv = torch.argsort(perm)
        for t in range(plan.num_tiles):
            pos, _ = window_keys(lat, tile, win, t)
            keys = torch.cat([perm[pos], text])
            mine = [i for i, r in enumerate(rows.tolist()) if r < S and int(inv[r]) // plan.tile_tokens == t]
            if mine:
                a, b_, _ = reference(Group(q[0, h, rows[mine]], k[0, h, keys], v[0, h, keys], [(0, len(keys))],
                                           None, "s"))
                want_s[mine], bound_s[mine] = a, b_
        tx = [where[int(r)] for r in text]
        want_s[tx], bound_s[tx] = full[0][tx], full[1][tx]          # text queries attend every valid key
        ref.append((want_s, bound_s))
        we = w[0, h].double()
        want = sum(we[e] * ref[e][0] for e in range(3))
        bound = sum(we[e] * ref[e][1] for e in range(3)) + U * want.abs()
        worst = max(worst, assert_within_bound(out[h, rows], want, bound, torch.zeros_like(want, dtype=torch.bool),
                                               f"blend head {h} std {std}"))
    report(f"peaked blend std {std}", worst)
