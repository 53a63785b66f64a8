"""Exact probes of how the attention kernel consumes its plan tables: which keys each query row attends to, where each
result row is written, and what a call must leave untouched.

The parity tests compare randn inputs with a cosine / max-abs bar, which cannot see one key too many or too few in a
window of thousands, nor a write outside the rows a call owns.  The inputs here are built so that the exact answer is
known and an error of one key or one row shows:

* key-set probe: Q lives in channels [0, 64) and K in [64, 128), so every logit is exactly 0 and the softmax is the
  uniform mean over the attended keys.  V holds small integer codes (balanced +-1 signs per tile and per text block,
  tile-coordinate buckets, a constant), so the sums are exact in fp32 and one missing, extra or substituted key moves
  an exact 0 or a small-count ratio by more than one bf16 ulp.  The CPU self-checks below prove that for every
  geometry, without a GPU.
* row-destination probe: Q = K = 64 * (random unit rows), so a query's own key beats every other logit by more than
  100 nats and the output row is exactly the V row of the query's own key (coreset: of its unpool source).
* output fence: the output is an interior view of a buffer filled with a bf16 NaN pattern; everything the call does
  not own must still hold it afterwards.
"""
import pytest
import torch

from oracle import vorta_oracle as O
from vorta_b200 import _lib as L
from vorta_b200 import ops

gpu = pytest.mark.gpu

SENTINEL = 0x7FA1          # a bf16 NaN: no attention output has these bits
ALPHA = 64.0               # |q| = |k|: self logit 4096 / sqrt(128) = 362, others below 0.45 of it
N_SIGN = 100               # channels [0, 100): balanced signs; [100, 112): tile buckets; 112: text; 127: constant
PAD_CODE = 37.0            # every channel of a padded text key: cannot cancel

# (latent, tile, window, lowres window, text_len, text_valid): the five cases of test_branches_vs_oracle (120-, 216-,
# 72- and 8-token tiles, a window larger than the grid), then the text edges TV == 0 and S + TV = 1 (mod 128)
GEOMS = [
    ((10, 12, 16), (5, 6, 4), (3, 3, 3), (2, 3, 2), 0, 0),
    ((6, 18, 16), (3, 9, 8), (3, 3, 3), (3, 3, 2), 0, 0),
    ((4, 9, 16), (1, 9, 8), (3, 1, 3), (1, 3, 4), 0, 0),
    ((6, 12, 8), (3, 6, 4), (3, 3, 3), (2, 3, 2), 40, 23),
    ((2, 4, 8), (1, 2, 4), (5, 5, 5), (2, 2, 2), 8, 8),
    ((6, 12, 8), (3, 6, 4), (3, 3, 3), (2, 3, 2), 40, 0),
    ((6, 12, 8), (3, 6, 4), (3, 3, 3), (2, 3, 2), 80, 65),   # S + TV = 641: the last key block holds one key
]
GEOM_IDS = ["tile120", "tile216", "tile72-asym", "text40-23", "window-over-grid", "text40-0", "last-block-1-key"]
WAN14 = ((21, 45, 80), (3, 9, 16), (3, 3, 3), (3, 3, 2), 0, 0)
WAN13 = ((21, 30, 52), (3, 10, 4), (3, 3, 3), (3, 3, 2), 0, 0)
HUNYUAN = ((33, 45, 80), (3, 9, 16), (3, 3, 3), (3, 3, 2), 256, 64)


def dev():
    L.check(L.lib().vb_device_check())
    return torch.device("cuda:0")


def to_dev(x, layout="token"):
    """(B, H, N, D) host tensor -> bf16 device view over (B, N, H, D) memory ("token") or (B, H, N, D) ("head")."""
    x = x.to(torch.bfloat16)
    if layout == "head":
        return x.contiguous().to(dev())
    return x.transpose(1, 2).contiguous().to(dev()).transpose(1, 2)


# ---------------------------------------------------------------------------------------------------------
# the bar: within one bf16 ulp of the fp64 answer, exactly 0 where it is 0
# ---------------------------------------------------------------------------------------------------------
def ulp_failures(got, want):
    got, want = got.double(), want.double()
    zero = want == 0
    ulp = torch.exp2(torch.floor(torch.log2(want.abs().clamp_min(1e-300))) - 7)
    return (zero & (got != 0)) | (~zero & ((got - want).abs() > ulp)) | ~torch.isfinite(got)


def assert_within_one_ulp(got, want, what=""):
    bad = ulp_failures(got.float().cpu(), want)
    if bad.any():
        i = tuple(int(x) for x in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements beyond one bf16 ulp, first at {i}: "
                             f"got {float(got.float().cpu()[i])}, want {float(want[i])}")


# ---------------------------------------------------------------------------------------------------------
# key-set probe inputs
# ---------------------------------------------------------------------------------------------------------
def balanced_signs(n_blocks, size, channels, g):
    """(n_blocks, size, channels) integer codes in {-1, 0, +1} summing to 0 over every block: half +1, half -1 in a
    random order per channel, and one 0 when the block is odd."""
    order = torch.rand((n_blocks, size, channels), generator=g, dtype=torch.float64).argsort(dim=1).argsort(dim=1)
    s = torch.where(order < size // 2, 1.0, -1.0).double()
    if size % 2:
        s[order == size - 1] = 0.0
    return s


def key_code(lat, tile, tl, tv, g):
    """V codes (S + tl, 128) float64 of one (batch, head), keys in raster order."""
    S = lat[0] * lat[1] * lat[2]
    tau = tile[0] * tile[1] * tile[2]
    nt = [lat[d] // tile[d] for d in range(3)]
    n_tiles = nt[0] * nt[1] * nt[2]
    perm = O.tile_permutation(lat, tile)                             # tile-major position -> raster token
    code = torch.zeros((S + tl, 128), dtype=torch.float64)
    code[perm, :N_SIGN] = balanced_signs(n_tiles, tau, N_SIGN, g).reshape(S, N_SIGN)
    t = torch.arange(n_tiles)
    coords = [t // (nt[1] * nt[2]), (t // nt[2]) % nt[1], t % nt[2]]
    bucket = torch.zeros((n_tiles, 12), dtype=torch.float64)
    for d in range(3):
        bucket[t, 4 * d + coords[d] % 4] = 1.0
    code[perm, N_SIGN:N_SIGN + 12] = bucket.repeat_interleave(tau, dim=0)
    if tv:
        code[S:S + tv, :N_SIGN] = balanced_signs(1, tv, N_SIGN, g)[0]
        code[S:S + tv, N_SIGN + 12] = 1.0
    code[:S + tv, 127] = 1.0
    code[S + tv:] = PAD_CODE
    return code


def uniform_logit_qkv(B, H, lat, tile, tl, tv, seed):
    """Q in channels [0, 64), K in [64, 128) (every logit exactly 0), V the key codes; float64 host tensors holding bf16
    values."""
    S = lat[0] * lat[1] * lat[2]
    g = torch.Generator().manual_seed(seed)
    q = torch.zeros((B, H, S + tl, 128), dtype=torch.float64)
    k = torch.zeros_like(q)
    q[..., :64] = torch.randn((B, H, S + tl, 64), generator=g, dtype=torch.float64)
    k[..., 64:] = torch.randn((B, H, S + tl, 64), generator=g, dtype=torch.float64)
    q, k = q.to(torch.bfloat16).double(), k.to(torch.bfloat16).double()
    v = torch.stack([torch.stack([key_code(lat, tile, tl, tv, g) for _ in range(H)]) for _ in range(B)])
    return q, k, v


def window_keys(lat, tile, win, t):
    """Tile-major key positions of query tile t's window (sorted), from the oracle's closed form."""
    nt = [lat[d] // tile[d] for d in range(3)]
    tau = tile[0] * tile[1] * tile[2]
    w = O.tile_windows(lat, win, tile)[t]
    ids = [(a * nt[1] + b) * nt[2] + c for a in range(w[0], w[3] + 1) for b in range(w[1], w[4] + 1)
           for c in range(w[2], w[5] + 1)]
    return torch.cat([torch.arange(i * tau, (i + 1) * tau) for i in sorted(ids)]), ids


# ---------------------------------------------------------------------------------------------------------
# C. sensitivity self-check (CPU): the bar rejects a key set off by one key, one 16-key step, one tile
# ---------------------------------------------------------------------------------------------------------
def _runs(pos):
    """Maximal contiguous runs [start, end) of sorted key positions."""
    cut = (torch.nonzero(pos[1:] != pos[:-1] + 1).flatten() + 1).tolist()
    bounds = [0] + cut + [len(pos)]
    return [(int(pos[a]), int(pos[b - 1]) + 1) for a, b in zip(bounds[:-1], bounds[1:])]


def _perturbations(pos, n_keys, S, tv, tl, tile_swap=None):
    """Key sets (kernel-order positions; video tile-major, then text) one mistake away from `pos`."""
    out = {}
    runs = _runs(pos)
    s0, e0 = runs[0]
    out["drop last key of a run"] = pos[pos != e0 - 1]
    past = [e for _, e in runs if e < n_keys and not bool((pos == e).any())]
    if past:
        out["add first key past a run end"] = torch.cat([pos, torch.tensor([past[0]])])
    tail = s0 + ((e0 - s0 - 1) // 128) * 128
    step = torch.arange(tail, min(tail + 16, e0))
    out["drop a 16-key step of a tail block"] = pos[~torch.isin(pos, step)]
    if tile_swap is not None:
        out["swap a window tile for its neighbour"] = tile_swap
    if tl > tv:
        out["include one padded text key"] = torch.cat([pos, torch.tensor([S + tv])])
    return out


def _neighbour_swap(lat, tile, win, t, pos):
    nt = [lat[d] // tile[d] for d in range(3)]
    tau = tile[0] * tile[1] * tile[2]
    w = O.tile_windows(lat, win, tile)[t]
    for d in range(3):
        for inside, outside in ((w[d], w[d] - 1), (w[3 + d], w[3 + d] + 1)):
            if 0 <= outside < nt[d]:
                lo = list(w[:3])
                lo[d] = inside
                a = [int(x) for x in lo]
                b = list(a)
                b[d] = outside
                old = (a[0] * nt[1] + a[1]) * nt[2] + a[2]
                new = (b[0] * nt[1] + b[1]) * nt[2] + b[2]
                keep = pos[(pos < old * tau) | (pos >= (old + 1) * tau)]
                return torch.cat([keep, torch.arange(new * tau, (new + 1) * tau)])
    return None            # the window covers the whole grid


def _mean_over(code_kernel_order, pos):
    return code_kernel_order[pos].mean(dim=0)


def _kernel_order(lat, tile, code):
    S = lat[0] * lat[1] * lat[2]
    perm = O.tile_permutation(lat, tile)
    return torch.cat([code[perm], code[S:]])


@pytest.mark.parametrize("geom", GEOMS + [WAN14], ids=GEOM_IDS + ["wan14"])
def test_key_set_bar_rejects_every_one_key_mistake(geom):
    """For every geometry of the key-set probe: the V codes averaged over the oracle's key set pass the bar, and the
    same codes averaged over each perturbed key set (rounded to bf16, as a kernel would write them) fail it."""
    lat, tile, win, lw, tl, tv = geom
    S = lat[0] * lat[1] * lat[2]
    g = torch.Generator().manual_seed(S + tl)
    code = _kernel_order(lat, tile, key_code(lat, tile, tl, tv, g))
    n_tiles = S // (tile[0] * tile[1] * tile[2])
    text = torch.arange(S, S + tv)
    cases = []
    for t in sorted({0, n_tiles // 2, n_tiles - 1}):                    # sliding: corner, interior, last tile
        pos, _ = window_keys(lat, tile, win, t)
        pos = torch.cat([pos, text])
        cases.append((f"sliding tile {t}", pos, _neighbour_swap(lat, tile, win, t, pos)))
    cases.append(("full", torch.arange(S + tv), None))
    checked = 0
    for name, pos, swap in cases:
        want = _mean_over(code, pos)
        assert not ulp_failures(want.to(torch.bfloat16).double(), want).any(), name
        for what, bad in _perturbations(pos, S + tv, S, tv, tl, swap).items():
            got = _mean_over(code, bad).to(torch.bfloat16).double()
            assert ulp_failures(got, want).any(), f"{name}: the bar accepts '{what}'"
            checked += 1
    assert checked >= 2 * len(cases)


def test_key_set_bar_rejects_dense_tail_mistakes():
    """Dense attention: one key fewer or more at the end of the key range fails the bar at every tested length."""
    g = torch.Generator().manual_seed(1)
    for n_k in (1, 15, 16, 17, 127, 128, 129, 257, 512):
        code = dense_key_code(n_k, g)
        want = code[:n_k].mean(dim=0)
        assert not ulp_failures(want.to(torch.bfloat16).double(), want).any()
        assert ulp_failures(code[:n_k + 1].mean(dim=0).to(torch.bfloat16).double(), want).any(), n_k
        if n_k > 1:
            assert ulp_failures(code[:n_k - 1].mean(dim=0).to(torch.bfloat16).double(), want).any(), n_k


def dense_key_code(n_k, g, extra=8):
    """(n_k + extra, 128): balanced signs over the n_k keys, a constant, then `extra` rows past the end that must never be
    read (PAD_CODE in every channel)."""
    code = torch.zeros((n_k + extra, 128), dtype=torch.float64)
    code[:n_k, :N_SIGN] = balanced_signs(1, n_k, N_SIGN, g)[0]
    code[:n_k, 127] = 1.0
    code[n_k:] = PAD_CODE
    return code


# ---------------------------------------------------------------------------------------------------------
# A. key-set probe on the GPU
# ---------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_every_row_attends_exactly_its_key_set(geom):
    lat, tile, win, lw, tl, tv = geom
    S = lat[0] * lat[1] * lat[2]
    B, H, layout = (2, 3, "head") if tl == 0 else (1, 3, "token")
    q, k, v = uniform_logit_qkv(B, H, lat, tile, tl, tv, seed=S + tl + tv)
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    info = O.get_group_info(lat, lw, 0.5)
    kv_from_k = tl > 0
    flags = L.ATTN_CORESET_KV_FROM_K if kv_from_k else 0
    qd, kd, vd = to_dev(q, layout), to_dev(k, layout), to_dev(v, layout)
    oracle = dict(text_len=tl, text_valid=tv, kv_from_k=kv_from_k)
    for branch in ([0] * H, [1] * H, [2] * H, [0, 1, 2]):
        out = ops.routed_attention(plan, qd, kd, vd, branch=branch, flags=flags)
        want = O.routed_attention(q, k, v, info, lat, win, tile, branch=torch.tensor(branch), **oracle)
        assert_within_one_ulp(out, want, f"branch {branch}")
    w = torch.softmax(torch.randn((B, H, 3), generator=torch.Generator().manual_seed(S)), -1)
    out = ops.routed_attention(plan, qd, kd, vd, weights=w, flags=flags)
    want = O.routed_attention(q, k, v, info, lat, win, tile, weights=w.double(), **oracle)
    assert_within_one_ulp(out, want, "blend")


@gpu
def test_wan14_key_sets_corner_edge_interior_tiles():
    """Wan-14B tiles of 432 tokens (48-row query tails, 16-key run tails): every full-head row is the mean over all
    keys, every coreset row the mean over the kept keys, and corner, edge and interior sliding tiles the mean over
    their oracle window."""
    lat, tile, win, lw, tl, tv = WAN14
    S = lat[0] * lat[1] * lat[2]
    q, k, v = uniform_logit_qkv(1, 3, lat, tile, 0, 0, seed=14)
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    out = ops.routed_attention(plan, to_dev(q), to_dev(k), to_dev(v), branch=[0, 1, 2]).float().cpu()
    assert_within_one_ulp(out[0, 0], v[0, 0].mean(dim=0).expand(S, 128), "full head")
    info = O.get_group_info(lat, lw, 0.5)
    m = O.match(q[:, 1:2], info)
    kept = torch.cat([info.center_indices[:, 0], O.kept_token_ids(info, m[0])[0, 0]])
    assert_within_one_ulp(out[0, 1], v[0, 1, kept].mean(dim=0).expand(S, 128), "coreset head")
    perm = O.tile_permutation(lat, tile)
    for t in (0, 4, 79, 87, 174):
        pos, _ = window_keys(lat, tile, win, t)
        rows = perm.reshape(-1, plan.tile_tokens)[t]
        want = v[0, 2, perm[pos]].mean(dim=0).expand(len(rows), 128)
        assert_within_one_ulp(out[0, 2, rows], want, f"sliding tile {t}")


@gpu
@pytest.mark.parametrize("heads", [3, 72])
def test_dense_rows_attend_exactly_their_keys(heads):
    """Dense attention with uniform logits: each row is the mean over exactly n_k keys.  K and V are prefix views of
    longer allocations whose extra rows hold codes that would show if read."""
    g = torch.Generator().manual_seed(heads)
    for n_q in (1, 127, 128, 129, 257, 300):
        for n_k in (1, 15, 16, 17, 127, 128, 129, 257, 512):
            q = torch.zeros((1, heads, n_q, 128), dtype=torch.float64)
            q[..., :64] = torch.randn((1, heads, n_q, 64), generator=g, dtype=torch.float64)
            kk = torch.zeros((1, heads, n_k + 8, 128), dtype=torch.float64)
            kk[..., 64:] = torch.randn((1, heads, n_k + 8, 64), generator=g, dtype=torch.float64)
            vv = torch.stack([dense_key_code(n_k, g) for _ in range(heads)])[None]
            kd, vd = to_dev(kk), to_dev(vv)
            out = ops.attn_dense(to_dev(q), kd[:, :, :n_k], vd[:, :, :n_k])
            want = vv[:, :, :n_k].mean(dim=2, keepdim=True).expand(1, heads, n_q, 128)
            assert_within_one_ulp(out, want, f"n_q {n_q}, n_k {n_k}")


# ---------------------------------------------------------------------------------------------------------
# B. row-destination probe
# ---------------------------------------------------------------------------------------------------------
def self_qkv(B, H, N, seed):
    """Q = K = ALPHA * random unit rows, V positive bf16 (no two rows alike); bf16 host tensors."""
    g = torch.Generator().manual_seed(seed)
    u = torch.randn((B, H, N, 128), generator=g)
    qk = (ALPHA * u / u.norm(dim=-1, keepdim=True)).to(torch.bfloat16)
    v = torch.exp2(torch.rand((B, H, N, 128), generator=g) * 3 - 1).to(torch.bfloat16)
    return qk, v


def self_sources(qk, branch_of_head, lat, lw, tl, tv):
    """(B, H, N) int64: the V row each output row must equal, -1 where the row must be 0 (padded text)."""
    B, H, N, _ = qk.shape
    S = N - tl
    src = torch.arange(N).repeat(B, H, 1)
    src[:, :, S + tv:] = -1
    info = None
    for h, e in enumerate(branch_of_head):
        if e != L.BRANCH_CORESET:
            continue
        info = info or O.get_group_info(lat, lw, 0.5)
        m = O.match(qk[:, h:h + 1, :S].double(), info)
        ids = torch.arange(S, dtype=torch.float64).view(1, 1, S, 1).expand(B, 1, S, 1)
        src[:, h, :S] = O.unpool(O.pool(ids, info, m), info, m)[:, 0, :, 0].long()
    return src


def rows_of(v, src):
    """v[b, h, src[b, h, i]] with zero rows where src < 0 (device or host)."""
    idx = src.clamp_min(0).to(v.device)[..., None].expand(-1, -1, -1, 128)
    return torch.where((src >= 0).to(v.device)[..., None], torch.gather(v, 2, idx), torch.zeros((), dtype=v.dtype,
                                                                                                device=v.device))


def assert_rows_equal(out, want, what=""):
    same = (out.view(torch.int16) == want.view(torch.int16)).all(dim=-1)
    if not bool(same.all()):
        i = tuple(int(x) for x in (~same).nonzero()[0])
        raise AssertionError(f"{what}: {int((~same).sum())} rows differ, first (b, h, row) = {i}")


def _self_probe(geom, B, H, branches, layout, seed, blend=True):
    lat, tile, win, lw, tl, tv = geom
    S = lat[0] * lat[1] * lat[2]
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    flags = L.ATTN_CORESET_KV_FROM_K if tl else 0
    qk, v = self_qkv(B, H, S + tl, seed)
    qd, vd = to_dev(qk, layout), to_dev(v, layout)
    for branch in branches:
        out = ops.routed_attention(plan, qd, qd, vd, branch=branch, flags=flags)
        assert_rows_equal(out, rows_of(vd, self_sources(qk, branch, lat, lw, tl, tv)), f"branch {branch}")
    if blend:
        w = torch.softmax(torch.randn((B, H, 3), generator=torch.Generator().manual_seed(seed)), -1)
        out = ops.routed_attention(plan, qd, qd, vd, weights=w, flags=flags)
        v64 = v.double()
        want = sum(w[:, :, e, None, None].double() * rows_of(v64, self_sources(qk, [e] * H, lat, lw, tl, tv))
                   for e in range(3))
        assert_within_one_ulp(out, want, "blend")


@gpu
@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_every_row_lands_at_its_destination(geom):
    S = geom[0][0] * geom[0][1] * geom[0][2]
    B, layout = (2, "head") if S % 3 == 0 else (1, "token")
    _self_probe(geom, B, 3, ([0] * 3, [1] * 3, [2] * 3, [0, 1, 2], [2, 0, 1]), layout, seed=S + geom[4])


@gpu
@pytest.mark.parametrize("geom", [WAN13, WAN14, HUNYUAN], ids=["wan13", "wan14", "hunyuan"])
def test_every_row_lands_at_its_destination_full_size(geom):
    _self_probe(geom, 1, 3, ([0, 1, 2],), "token", seed=7, blend=False)


@gpu
@pytest.mark.parametrize("heads", [3, 72])
def test_dense_rows_land_at_their_destination(heads):
    g = torch.Generator().manual_seed(100 + heads)
    for n_q in (1, 127, 128, 129, 257, 300):
        for n_k in (1, 15, 16, 17, 127, 128, 129, 257, 512):
            k, v = self_qkv(1, heads, n_k, seed=int(torch.randint(1 << 30, (1,), generator=g)))
            src = (torch.arange(n_q) % n_k).repeat(1, heads, 1)
            kd, vd = to_dev(k), to_dev(v)
            out = ops.attn_dense(kd[:, :, src[0, 0]], kd, vd)
            assert_rows_equal(out, rows_of(vd, src), f"n_q {n_q}, n_k {n_k}")


# ---------------------------------------------------------------------------------------------------------
# D. output fence
# ---------------------------------------------------------------------------------------------------------
GUARD = 3


def fenced(B, H_out, N):
    """A sentinel-filled buffer and the (B, H_out, N, 128) output view inside it: guard rows before and after, a head
    on either side and a padded batch stride."""
    buf = torch.full((B, N + 2 * GUARD + 5, H_out + 2, 128), SENTINEL, dtype=torch.int16, device=dev())
    return buf, buf.view(torch.bfloat16)[:, GUARD:GUARD + N, 1:1 + H_out].transpose(1, 2)


def assert_fence(buf, owned, N, what=""):
    """Every element outside `owned` (B, H_out, N) still holds the sentinel."""
    mask = torch.zeros(buf.shape[:3], dtype=torch.bool, device=buf.device)
    mask[:, GUARD:GUARD + N, 1:1 + owned.shape[1]] = owned.transpose(1, 2).to(buf.device)
    hit = (buf != SENTINEL).any(dim=-1) & ~mask
    if bool(hit.any()):
        i = tuple(int(x) for x in hit.nonzero()[0])
        raise AssertionError(f"{what}: {int(hit.sum())} rows written outside the call's rows, first (b, buffer row, "
                             f"buffer head) = {i}")


TEXT = GEOMS[3]


def _plan_and_inputs(geom, H, seed):
    lat, tile, win, lw, tl, tv = geom
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    qk, v = self_qkv(1, H, plan.seq_len + tl, seed)
    return plan, qk, v, to_dev(qk), to_dev(v)


@gpu
def test_fence_top1_out_heads_with_text():
    """Top-1 heads {5, 1, 6} of an 8-head output with padded text: only those heads' rows, padded rows zeroed."""
    lat, tile, win, lw, tl, tv = TEXT
    plan, qk, v, qd, vd = _plan_and_inputs(TEXT, 3, 31)
    N, mine, branch = plan.seq_len + tl, [5, 1, 6], [0, 1, 2]
    buf, out = fenced(1, 8, N)
    ops.routed_attention(plan, qd, qd, vd, branch=branch, flags=L.ATTN_CORESET_KV_FROM_K, out=out, out_heads=mine)
    owned = torch.zeros((1, 8, N), dtype=torch.bool)
    owned[:, mine] = True
    assert_fence(buf, owned, N, "top-1")
    assert_rows_equal(out[:, mine], rows_of(vd, self_sources(qk, branch, lat, lw, tl, tv)), "top-1")


@gpu
def test_fence_skip_slots_write_nothing():
    """SKIP slots (padding of a rank's slot table, out_heads 0) own no rows, padded text rows included."""
    lat, tile, win, lw, tl, tv = TEXT
    plan, qk, v, qd, vd = _plan_and_inputs(TEXT, 5, 32)
    N = plan.seq_len + tl
    branch, dest = [1, L.BRANCH_SKIP, 0, L.BRANCH_SKIP, 2], [3, 0, 0, 0, 1]
    buf, out = fenced(1, 4, N)
    ops.routed_attention(plan, qd, qd, vd, branch=branch, flags=L.ATTN_CORESET_KV_FROM_K, out=out, out_heads=dest)
    owned = torch.zeros((1, 4, N), dtype=torch.bool)
    owned[:, [3, 0, 1]] = True
    assert_fence(buf, owned, N, "skip slots")
    live = [0, 2, 4]
    want = rows_of(vd[:, live], self_sources(qk[:, live], [branch[i] for i in live], lat, lw, tl, tv))
    assert_rows_equal(out[:, [3, 0, 1]], want, "skip slots")


@gpu
@pytest.mark.parametrize("geom", [TEXT, GEOMS[1]], ids=["text40-23", "tile216"])
def test_fence_query_parts_own_disjoint_rows(geom):
    """Each query part of a full head, run alone, writes whole rows of its own head only; the parts' rows are disjoint
    and their union is every row of the head (halves and quarters)."""
    lat, tile, win, lw, tl, tv = geom
    plan, qk, v, qd, vd = _plan_and_inputs(geom, 1, 33)
    N = plan.seq_len + tl
    want = rows_of(vd, self_sources(qk, [0], lat, lw, tl, tv))
    for parts in ([L.BRANCH_FULL_LO, L.BRANCH_FULL_HI], [L.branch_full_part(i, 4) for i in (2, 0, 3, 1)]):
        cover = torch.zeros(N, dtype=torch.int32)
        for e in parts:
            buf, out = fenced(1, 2, N)
            ops.routed_attention(plan, qd, qd, vd, branch=[e], out=out, out_heads=[1])
            written = (out[0, 1].view(torch.int16) != SENTINEL).any(dim=-1).cpu()
            owned = torch.zeros((1, 2, N), dtype=torch.bool)
            owned[0, 1] = written
            assert_fence(buf, owned, N, f"part {e}")
            assert bool((out[0, 1].view(torch.int16) != SENTINEL).all(dim=-1).cpu()[written].all()), f"part {e}"
            assert_rows_equal(out[:, 1:2, written], want[:, :, written], f"part {e}")
            cover += written.int()
        assert bool((cover == 1).all()), f"parts {parts}: rows covered {cover.unique().tolist()} times"
    # all parts and a whole head in one launch, out of order
    buf, out = fenced(1, 2, N)
    ids = [L.branch_full_part(2, 4), 0, L.branch_full_part(0, 4), L.branch_full_part(3, 4), L.branch_full_part(1, 4)]
    ops.routed_attention(plan, qd[:, [0] * 5], qd[:, [0] * 5], vd[:, [0] * 5], branch=ids, out=out,
                         out_heads=[1, 0, 1, 1, 1])
    assert_fence(buf, torch.ones((1, 2, N), dtype=torch.bool), N, "quarters + whole head")
    assert_rows_equal(out, torch.cat([want, want], dim=1), "quarters + whole head")


@gpu
def test_blend_with_out_heads_equals_plain_blend():
    """Blend mode into heads {5, 1, 6} of an 8-head output gives the bits of the same blend into its own output, and
    leaves the other heads alone (the fp32 accumulator follows the head slots, not the output's head index)."""
    lat, tile, win, lw, tl, tv = TEXT
    plan, qk, v, qd, vd = _plan_and_inputs(TEXT, 3, 34)
    N, mine = plan.seq_len + tl, [5, 1, 6]
    w = torch.softmax(torch.randn((1, 3, 3), generator=torch.Generator().manual_seed(34)), -1)
    plain = ops.routed_attention(plan, qd, qd, vd, weights=w, flags=L.ATTN_CORESET_KV_FROM_K)
    out = torch.full((1, N, 8, 128), SENTINEL, dtype=torch.int16, device=dev())
    ops.routed_attention(plan, qd, qd, vd, weights=w, flags=L.ATTN_CORESET_KV_FROM_K,
                         out=out.view(torch.bfloat16).transpose(1, 2), out_heads=mine)
    rest = [h for h in range(8) if h not in mine]
    assert bool((out[:, :, rest] == SENTINEL).all()), "blend wrote other heads"
    assert torch.equal(out[:, :, mine], plain.transpose(1, 2).view(torch.int16))


@gpu
def test_fence_dense_strided_view():
    k, v = self_qkv(2, 3, 129, seed=35)
    src = (torch.arange(300) % 129).repeat(2, 3, 1)
    kd, vd = to_dev(k, "head"), to_dev(v, "head")
    buf, out = fenced(2, 3, 300)
    ops.attn_dense(kd[:, :, src[0, 0]], kd, vd, out=out)
    assert_fence(buf, torch.ones((2, 3, 300), dtype=torch.bool), 300, "dense")
    assert_rows_equal(out, rows_of(vd, src), "dense")


# ---------------------------------------------------------------------------------------------------------
# E. argument validation: every malformed shape is refused before a launch (prefix views of real memory, so the call
# could not fault even where the check were missing)
# ---------------------------------------------------------------------------------------------------------
@gpu
def test_routed_attention_refuses_mismatched_output_and_out_heads():
    lat, tile, win, lw, tl, tv = TEXT
    plan, qk, v, qd, vd = _plan_and_inputs(TEXT, 3, 36)
    N = plan.seq_len + tl
    big = torch.zeros((2, N + 8, 8, 128), dtype=torch.bfloat16, device=dev()).transpose(1, 2)
    run = lambda **kw: ops.routed_attention(plan, qd, qd, vd, branch=[0, 1, 2], flags=L.ATTN_CORESET_KV_FROM_K, **kw)
    with pytest.raises(ValueError):
        run(out=big[:1, :3, :N - 1])                           # too few rows
    with pytest.raises(ValueError):
        run(out=big[:1, :3, :N + 1])                           # too many rows
    with pytest.raises(ValueError):
        run(out=big[:, :3, :N])                                # batch 2 for a batch-1 call
    with pytest.raises(ValueError):
        run(out=big[:1, :2, :N])                               # fewer heads than the call writes
    with pytest.raises(ValueError):
        run(out=big[:1, :6, :N], out_heads=[5, 1, 6])          # head 6 of a 6-head output
    with pytest.raises(ValueError):
        run(out=big[:1, :, :N], out_heads=[5, 1])              # one output head per local head
    with pytest.raises(ValueError):
        ops.routed_attention(plan, qd, qd, vd[:, :2], branch=[0, 1, 2])
    run(out=big[:1, :7, :N], out_heads=[5, 1, 6])              # the smallest output that holds head 6


@gpu
def test_attn_dense_refuses_mismatched_keys_values_and_output():
    g = torch.Generator().manual_seed(37)
    q = to_dev(torch.randn((2, 3, 100, 128), generator=g), "head")
    kv = to_dev(torch.randn((2, 3, 77, 128), generator=g), "head")
    with pytest.raises(ValueError):
        ops.attn_dense(q, kv, kv[:, :, :60])                   # k and v lengths differ
    with pytest.raises(ValueError):
        ops.attn_dense(q, kv[:, :2], kv[:, :2])                # fewer heads than q
    with pytest.raises(ValueError):
        ops.attn_dense(q, kv[:1], kv[:1])                      # fewer batch elements than q
    with pytest.raises(ValueError):
        ops.attn_dense(q, kv, kv, out=torch.empty_like(q)[:, :, :99])
    ops.attn_dense(q, kv, kv, out=torch.empty_like(q))
