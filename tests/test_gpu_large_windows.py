"""Large coreset windows (groups of more than 33 tokens, which the shared-memory selection kernel runs) and sliding
windows of more than 32 key runs per window group, on the GPU against the pinned CPU oracle.

The reference's goldens cover none of these geometries and none can be made without the reference's code; the oracle
(held to those goldens by tests/test_oracle_golden.py) is the reference.  Index tables are compared with the oracle's
``match`` run in fp64, the ranking the selection kernels promise (DESIGN.md section 3.3); attention outputs at the bar
of tests/test_gpu_parity.py; softmax weights at the fp64 bar of tests/test_gpu_attn_numerics.py."""
import pytest
import torch

from oracle import fixtures as FX
from oracle import vorta_oracle as O
from oracle.make_golden import fullsize_coreset_input
from vorta_b200 import _lib as L
from vorta_b200 import ops

from test_gpu_attn_numerics import _peaked, report
from test_gpu_parity import assert_attn_close, dev, to_dev_bhnd

pytestmark = pytest.mark.gpu

GROUP_WINDOWS = [(1, 6, 6), (2, 4, 6), (4, 4, 4), (2, 6, 6), (2, 8, 8), (4, 8, 8)]     # g = 36 .. 256
GROUP_LATENT = (8, 24, 24)


def _gid(w):
    return f"g{w[0] * w[1] * w[2]}"


def _match_fp64(x, info):
    """The oracle's ``match`` in fp64 with its ties broken the kernels' way, lower margin position first (a stable
    ascending sort of the same similarities; ``match``'s argsort orders exact ties arbitrarily)."""
    order = torch.sort(O.similarity(x.double(), info), dim=-1, stable=True).indices
    n_u = info.num_unpooled_tokens_per_group
    return order[..., :n_u], order[..., n_u:]


def _check_selection(plan, info, x):
    """Every table of vb_coreset_select against the fp64 oracle, and the partition property."""
    un, po, kept, drop = ops.coreset_select(plan, x.to(dev()), want_tokens=True)
    un_ref, po_ref = _match_fp64(x, info)
    assert torch.equal(un.cpu(), un_ref) and torch.equal(po.cpu(), po_ref)
    B, H = x.shape[:2]
    kept_ref = torch.cat([info.center_indices[:, 0].expand(B, H, -1), O.kept_token_ids(info, un_ref)], dim=-1)
    assert torch.equal(kept.cpu().long(), kept_ref)
    assert torch.equal(drop.cpu().long(), O.dropped_token_ids(info, po_ref))
    S = plan.seq_len
    for b in range(B):
        for h in range(H):
            allt = torch.cat([kept[b, h].cpu().long(), drop[b, h].cpu().long().flatten()])
            assert torch.equal(allt.sort().values, torch.arange(S))       # kept or dropped, exactly once


def _near_ties(x, info, seed):
    """Per group: an exact duplicate margin (a tie: the lower margin position ranks first), a pair whose cosines are
    about 1e-7 apart (one bf16 ulp in a channel of magnitude 2^-9), rows scaled by 2^-70 / 2^60 / 2^64 (fp32 squares
    underflow / stay finite / overflow), an all-zero margin and one tiny row among normal ones."""
    x = x.clone()
    bits = x.view(torch.int16)
    g = torch.Generator().manual_seed(seed)
    for grp in range(info.margin_indices.shape[0]):
        m = info.margin_indices[grp]
        n = m.numel()
        c = int(info.center_indices[grp, 0])
        a, b_, d, e = (int(i) for i in torch.randperm(n, generator=g)[:4])
        bits[:, :, m[b_]] = bits[:, :, m[a]]                              # exact tie
        bits[:, :, m[e]] = bits[:, :, m[d]]
        ch = int(torch.randint(0, 128, (1,), generator=g))
        x[:, :, m[d], ch] = 2.0 ** -9
        x[:, :, m[e], ch] = 2.0 ** -9
        bits[:, :, m[e], ch] += 1                                         # ~1e-7 apart
        rows = torch.cat([m, torch.tensor([c])])
        kind = grp % 8
        if kind == 1:
            x[:, :, rows] = (x[:, :, rows].float() * 2.0 ** -70).to(torch.bfloat16)
        elif kind == 2:
            x[:, :, rows] = (x[:, :, rows].float() * 2.0 ** 60).to(torch.bfloat16)
        elif kind == 3:
            x[:, :, rows] = (x[:, :, rows].float() * 2.0 ** 64).to(torch.bfloat16)
        elif kind == 4:
            x[:, :, m[(a + 1) % n]] = 0
        elif kind == 5:
            i = (a + 2) % n
            x[:, :, m[i]] = (x[:, :, m[i]].float() * 2.0 ** -70).to(torch.bfloat16)
    assert torch.isfinite(x.float()).all()
    return x


def _min_gap(x, info):
    """Smallest fp64 cosine gap between two different margins of a group (0 for exact ties)."""
    s = O.similarity(x.double(), info).sort(dim=-1).values
    return float((s[..., 1:] - s[..., :-1]).min())


# ---------------------------------------------------------------------------------------------------------
# index contract
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lw", GROUP_WINDOWS, ids=_gid)
def test_large_group_index_contract_vs_fp64_oracle(lw):
    plan = ops.Plan(GROUP_LATENT, (1, 1, 1), (1, 1, 1), lw, 0.5)
    info = O.get_group_info(GROUP_LATENT, lw, 0.5)
    g = plan.group_size
    _check_selection(plan, info, fullsize_coreset_input(GROUP_LATENT, 3, 100 + g))               # N(0, 1)
    smooth = fullsize_coreset_input(GROUP_LATENT, 3, 200 + g, smooth=0.05)                        # cosines 0.99+
    _check_selection(plan, info, smooth)
    x = _near_ties(fullsize_coreset_input(GROUP_LATENT, 2, 300 + g), info, g)
    assert _min_gap(x, info) == 0.0
    _check_selection(plan, info, x)


@pytest.mark.parametrize("lat,lw", [((6, 22, 4), (3, 11, 1)), ((4, 34, 4), (2, 17, 1))], ids=["g33", "g34"])
def test_kernel_boundary_matches_fp64_oracle(lat, lw):
    """g = 33 is the warp kernel's last group size (a margin per lane), g = 34 the shared-memory kernel's first: both
    equal the same fp64 oracle, near ties included, so which kernel ran a group does not show in its tables."""
    plan = ops.Plan(lat, (1, 1, 1), (1, 1, 1), lw, 0.5)
    info = O.get_group_info(lat, lw, 0.5)
    _check_selection(plan, info, fullsize_coreset_input(lat, 4, 33))
    _check_selection(plan, info, fullsize_coreset_input(lat, 4, 34, smooth=0.02))
    x = _near_ties(fullsize_coreset_input(lat, 4, 35), info, 35)
    gaps = O.similarity(x.double(), info).sort(dim=-1).values.diff(dim=-1)
    assert bool(((gaps > 0) & (gaps < 1e-6)).any())          # near ties below the fp32 bound, not only exact ones
    _check_selection(plan, info, x)


def test_largest_group_matches_fp64_oracle():
    """g = 4843, the largest group: one group over the grid, its similarities fill the opt-in shared memory."""
    lat = (29, 167, 1)
    plan = ops.Plan(lat, (1, 1, 1), (1, 1, 1), lat, 0.5)
    info = O.get_group_info(lat, lat, 0.5)
    _check_selection(plan, info, fullsize_coreset_input(lat, 3, 4843))
    _check_selection(plan, info, _near_ties(fullsize_coreset_input(lat, 2, 4844), info, 1))


# ---------------------------------------------------------------------------------------------------------
# branch outputs
# ---------------------------------------------------------------------------------------------------------
BRANCH_GEOMS = [   # (latent, tile, window, lowres window, heads, text_len, text_valid)
    ((12, 6, 8), (1, 2, 2), (13, 3, 3), (2, 3, 8), 3, 0, 0),       # g = 48, 36-run window groups
    ((12, 6, 8), (1, 2, 2), (13, 3, 3), (2, 3, 8), 3, 16, 11),     # + text: 37 runs, K's own matching for K / V
    ((8, 8, 8), (2, 2, 2), (3, 3, 3), (4, 4, 4), 2, 0, 0),         # g = 64
    ((8, 16, 16), (2, 4, 4), (3, 3, 3), (4, 8, 8), 2, 24, 24),     # g = 256 with text
    ((10, 20, 6), (1, 2, 2), (11, 11, 1), (2, 4, 6), 2, 8, 5),     # n < window: 101 runs; g = 48
]


@pytest.mark.parametrize("lat,tile,win,lw,H,tl,tv", BRANCH_GEOMS)
def test_large_window_branches_vs_oracle(lat, tile, win, lw, H, tl, tv):
    S = lat[0] * lat[1] * lat[2]
    g = torch.Generator().manual_seed(S + H + tl)
    q, k, v = (torch.randn((1, H, S + tl, 128), generator=g).to(torch.bfloat16) for _ in range(3))
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    info = O.get_group_info(lat, lw, 0.5)
    kv_from_k = tl > 0
    flags = L.ATTN_CORESET_KV_FROM_K if kv_from_k else 0
    qd, kd, vd = to_dev_bhnd(q), to_dev_bhnd(k), to_dev_bhnd(v)
    okw = dict(text_len=tl, text_valid=tv, kv_from_k=kv_from_k)
    for branch in ([1] * H, [2] * H, [h % 3 for h in range(H)]):
        out = ops.routed_attention(plan, qd, kd, vd, branch=branch, flags=flags)
        ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, win, tile, branch=torch.tensor(branch),
                                 **okw)
        assert_attn_close(out, ref)
    w = torch.softmax(torch.randn((1, H, 3), generator=g), dim=-1)
    out = ops.routed_attention(plan, qd, kd, vd, weights=w, flags=flags)
    ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, win, tile, weights=w, **okw)
    assert_attn_close(out, ref)


@pytest.mark.parametrize("lat,lw", [((8, 8, 8), (4, 4, 4)), ((8, 16, 16), (4, 8, 8)), ((12, 6, 8), (2, 3, 8))],
                         ids=lambda x: str(x))
def test_unpool_broadcast_one_hot_readout(lat, lw):
    """One-hot V (token t carries a 1 in channel t mod 128): a pooled row's output is its attention weights folded
    into 128 channels.  Every dropped margin (fp64 oracle's matching) holds its centre's row bit for bit, every kept
    token a row of its own, and the weights of every row sum to 1."""
    H = 2
    S = lat[0] * lat[1] * lat[2]
    plan = ops.Plan(lat, (1, 1, 1), (1, 1, 1), lw, 0.5)
    info = O.get_group_info(lat, lw, 0.5)
    gen = torch.Generator().manual_seed(S)
    q, k = (2.0 * torch.randn((1, H, S, 128), generator=gen) for _ in range(2))
    q, k = q.to(torch.bfloat16), k.to(torch.bfloat16)
    v = torch.zeros((1, H, S, 128))
    v[:, :, torch.arange(S), torch.arange(S) % 128] = 1.0
    v = v.to(torch.bfloat16)
    out = ops.routed_attention(plan, to_dev_bhnd(q), to_dev_bhnd(k), to_dev_bhnd(v), branch=[1] * H).cpu()
    un, po = O.match(q.double(), info)
    drop = O.dropped_token_ids(info, po)                                  # (1, H, G, n_p)
    kept = O.kept_token_ids(info, un)
    centres = info.center_indices[:, 0]
    bits = out.view(torch.int16)
    for h in range(H):
        c_rows = bits[0, h, centres]                                      # (G, 128)
        assert torch.equal(bits[0, h, drop[0, h]], c_rows[:, None].expand(-1, drop.shape[-1], -1))
        assert not torch.equal(bits[0, h, kept[0, h]], c_rows.repeat_interleave(kept.shape[-1] // len(centres), 0))
    sums = out.float().sum(-1)
    assert (sums - 1).abs().max().item() <= 2e-2
    ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, (1, 1, 1), (1, 1, 1),
                             branch=torch.tensor([1] * H))
    assert_attn_close(out, ref)


# ---------------------------------------------------------------------------------------------------------
# processors
# ---------------------------------------------------------------------------------------------------------
P_LAT, P_TILE, P_WIN, P_LW = (12, 6, 8), (1, 2, 2), (13, 3, 3), (2, 3, 8)


def _kwargs(text_len=0, text_valid=0):
    from vorta_b200.attention import create_sliding_tile_attn_mask_func, get_group_info
    d = dev()
    return dict(lowres_group_info=get_group_info(P_LAT, P_LW, 0.5, device=d),
                flex_attn_mask_func=create_sliding_tile_attn_mask_func(P_LAT, P_WIN, P_TILE, text_len, text_valid, d),
                window_size=P_WIN, tile_size=P_TILE, latent_shape=P_LAT)


def _oracle(q, k, v, **kw):
    info = O.get_group_info(P_LAT, P_LW, 0.5)
    return O.routed_attention(q.float().cpu(), k.float().cpu(), v.float().cpu(), info, P_LAT, P_WIN, P_TILE, **kw)


def test_wan_processors_with_large_windows():
    """Top-1 Eval (every branch on some head) and blend Train through the Wan processors."""
    from vorta_b200.attention import WanAttnProcessorTripleEval, WanAttnProcessorTripleTrain
    H = 3
    S = P_LAT[0] * P_LAT[1] * P_LAT[2]
    attn = FX.FakeWanAttn(H, seed=51).to(dev(), torch.bfloat16)
    attn32 = FX.FakeWanAttn(H, seed=51)
    hs = FX.det_tensor((1, S, H * 128), 52).to(dev(), torch.bfloat16)
    rot = FX.wan_rotary(S, 53).to(dev())
    kw = _kwargs()
    mix = torch.tensor(FX.MIX, device=dev())
    ev, tr = WanAttnProcessorTripleEval(check_input=True), WanAttnProcessorTripleTrain(check_input=True)
    q, k, v, _ = ev._input_proj(attn, hs, None, rot)

    def out_proj(o):
        with torch.no_grad():
            return attn32.to_out[0](o.transpose(1, 2).flatten(2, 3))

    with torch.no_grad():
        got_ev = ev(attn, hs, None, None, rot, tau_sparse=0.3, routing_score=mix, **kw)
        got_tr = tr(attn, hs, None, None, rot, routing_score=mix, **kw)
    ref_ev = out_proj(_oracle(q, k, v, branch=torch.tensor([0, 1, 2])))
    ref_tr = out_proj(_oracle(q, k, v, weights=mix.cpu()))
    scale = max(ref_ev.abs().max().item(), 1.0)
    assert_attn_close(got_ev, ref_ev, max_abs=2e-2 * scale)
    assert_attn_close(got_tr, ref_tr, max_abs=2e-2 * scale)


@pytest.mark.parametrize("dual", [True, False], ids=["dual-stream", "single-stream"])
def test_hunyuan_processors_with_large_windows_batch2_per_sample_text(dual):
    """HunyuanVideo Eval (routing from sample 0's scores, hunyuan.py:620-624) and Train at batch 1 and at batch 2 with
    per-sample text lengths: the attention output of every sample against the oracle with that sample's length, the
    padded text rows exactly zero, and the processor output of sample b equal to a batch-1 call within bf16
    tolerance."""
    from vorta_b200.attention import HunyuanVideoFlashAttnProcessorTripleEval, HunyuanVideoFlashAttnProcessorTripleTrain
    H, TL, TVS = 3, 24, [17, 5]
    S = P_LAT[0] * P_LAT[1] * P_LAT[2]
    d = dev()
    attn = FX.FakeHunyuanAttn(H, dual=dual, seed=61).to(d, torch.bfloat16)
    hs = FX.det_tensor((2, S, H * 128), 62).to(d, torch.bfloat16)
    ehs = FX.det_tensor((2, TL, H * 128), 63).to(d, torch.bfloat16)
    mask = torch.zeros(2, 1, 1, S + TL, dtype=torch.bool, device=d)
    for b, tv in enumerate(TVS):
        mask[b, ..., :S + tv] = True
    c, s = FX.hunyuan_rotary(S, 64)
    rope = (c.to(d), s.to(d))
    kw = _kwargs()
    kw["flex_attn_mask_func"] = None
    score = torch.softmax(FX.det_tensor((2, H, 3), 65, 4.0), -1).to(d)
    branch0 = O.route_top1(score.cpu(), 0.3)
    procs = {"eval": (HunyuanVideoFlashAttnProcessorTripleEval(check_input=True),
                      lambda sc: dict(kw, routing_score=sc, tau_sparse=0.3)),
             "train": (HunyuanVideoFlashAttnProcessorTripleTrain(check_input=True),
                       lambda sc: dict(kw, routing_score=sc))}
    for name, (proc, extra) in procs.items():
        with torch.no_grad():
            full_v, full_t = proc(attn, hs, ehs, mask, rope, **extra(score))
            q, k, v = proc._qkv(attn, hs, ehs, rope)
            proc._step_to_output = lambda attn_, vid, txt: (vid, txt)       # the attention output itself
            for B in (1, 2):
                att_v, att_t = proc(attn, hs[:B], ehs[:B], mask[:B], rope, **extra(score[:B]))
                for b in range(B):
                    okw = dict(text_len=TL, text_valid=TVS[b], kv_from_k=True)
                    if name == "eval":
                        okw["branch"] = branch0
                    else:
                        okw["weights"] = score[b:b + 1].cpu()
                    ref = _oracle(q[b:b + 1], k[b:b + 1], v[b:b + 1], **okw)
                    got = torch.cat([att_v[b:b + 1], att_t[b:b + 1]], dim=2)
                    assert_attn_close(got[:, :, :S + TVS[b]], ref[:, :, :S + TVS[b]])
                    assert torch.count_nonzero(att_t[b, :, TVS[b]:].float()) == 0, f"{name} B {B} sample {b}"
            del proc._step_to_output
            for b in range(2):
                sc = score[b:b + 1] if name == "train" else score[:1]
                one_v, one_t = proc(attn, hs[b:b + 1], ehs[b:b + 1], mask[b:b + 1], rope, **extra(sc))
                for got, want in ((full_v[b:b + 1], one_v), (full_t[b:b + 1], one_t)):
                    bad = (got.float() - want.float()).abs() > 0.02 + 0.02 * want.float().abs()
                    assert not bool(bad.any()), f"{name} sample {b}"


# ---------------------------------------------------------------------------------------------------------
# softmax weights at the fp64 bar
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("geom", [
    ((12, 6, 8), (1, 2, 2), (13, 3, 3), (2, 3, 8), 16, 11),        # g = 48 coreset, 37-run sliding window groups
    ((10, 20, 6), (1, 2, 2), (11, 11, 1), (2, 4, 6), 8, 5),        # 101 runs
    ((8, 16, 16), (2, 4, 4), (3, 3, 3), (4, 8, 8), 24, 24),        # g = 256 coreset
], ids=["g48-37runs", "101runs", "g256"])
def test_large_window_softmax_weights_fp64_bar(geom):
    """Full, coreset and sliding heads of one launch: sampled rows' softmax weights and outputs against fp64
    (test_gpu_attn_numerics._peaked at logit std 4)."""
    report(f"peaked large window {geom[0]} {geom[2]} {geom[3]}", _peaked(geom, 4.0, seed=9))


# ---------------------------------------------------------------------------------------------------------
# Wan DiT step
# ---------------------------------------------------------------------------------------------------------
def test_wan_dit_step_with_large_windows(monkeypatch):
    """A tiny Wan DiT step with a 48-token coreset window and 36-run sliding window groups, every branch routed on
    some head, against the fp32 torch restatement of the reference's block dataflow (tests/test_gpu_dit.py, same
    tolerance)."""
    import test_gpu_dit as D
    for name, val in (("LAT", P_LAT), ("TILE", P_TILE), ("WIN", P_WIN), ("LW", P_LW)):
        monkeypatch.setattr(D, name, val)
    D._wan_dit_step_check(dim=384, heads=3)
