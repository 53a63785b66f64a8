"""GPU parity tests: the sm_100a path, called through the C ABI, against (a) the golden vectors produced by the
reference's own code and (b) the CPU oracle on the same seeded inputs.

Bars (BASELINE.json): coreset indices, tile schedule, routing decisions — bit-exact; attention outputs —
cosine >= 0.999 and max-abs <= 2e-2 against the fp32 oracle.
"""
import numpy as np
import pytest
import torch

from oracle import fixtures as FX
from oracle import vorta_oracle as O
from vorta_b200 import _lib as L
from vorta_b200 import ops
from vorta_b200.attention import (HunyuanVideoFlashAttnProcessorTripleEval, HunyuanVideoFlashAttnProcessorTripleTrain,
                                  MatchingResults, WanAttnProcessor2_0, WanAttnProcessorTripleEval,
                                  WanAttnProcessorTripleTrain,
                                  create_sliding_tile_attn_mask_func, get_group_info, pool_sequence_by_similarity,
                                  sliding_tile_flex_attn, tile_layout, unpool_sequence_by_similarity, untile_layout)
from vorta_b200.patch import Router, route_step

pytestmark = pytest.mark.gpu

COS_MIN, MAX_ABS = 0.999, 2e-2          # BASELINE.json tolerance for attention outputs


def dev():
    L.check(L.lib().vb_device_check())
    return torch.device("cuda:0")


def assert_attn_close(out, ref, cos_min=COS_MIN, max_abs=MAX_ABS):
    out, ref = out.float().cpu(), ref.float().cpu()
    assert out.shape == ref.shape
    assert torch.isfinite(out).all()
    cos = torch.nn.functional.cosine_similarity(out.flatten(), ref.flatten(), dim=0).item()
    err = (out - ref).abs().max().item()
    assert cos >= cos_min, f"cosine {cos}"
    assert err <= max_abs, f"max-abs {err}"


def to_dev_bhnd(x):
    """(B, H, N, D) host tensor -> bf16 device view over (B, N, H, D) memory (the layout the projections produce)."""
    return x.to(torch.bfloat16).transpose(1, 2).contiguous().to(dev()).transpose(1, 2)


# ---------------------------------------------------------------------------------------------------------
# exact kernels
# ---------------------------------------------------------------------------------------------------------
def test_coreset_tables_bit_exact_vs_reference(golden):
    for rec in golden("coreset.pt"):
        plan = ops.Plan(rec["latent"], (1, 1, 1), (1, 1, 1), rec["window"], rec["rate"])
        un, po = ops.coreset_select(plan, rec["x"].to(dev()))
        assert un.dtype == torch.int64 and po.dtype == torch.int64
        # the kernel accumulates in fp64: equal to the reference run in fp64 ...
        assert torch.equal(un.cpu(), rec["unpooled_f64"])
        assert torch.equal(po.cpu(), rec["pooled_f64"])
        # ... and to the reference run in fp32 (the contract dtype) on these inputs
        assert torch.equal(un.cpu(), rec["unpooled_f32"])
        assert torch.equal(po.cpu(), rec["pooled_f32"])


def test_pool_unpool_bit_exact_vs_reference(golden):
    for rec in golden("coreset.pt"):
        info = get_group_info(rec["latent"], rec["window"], rec["rate"])
        x = rec["x"].to(dev())
        pooled, m = pool_sequence_by_similarity(x, info)
        assert torch.equal(pooled.cpu(), rec["pooled_seq"])
        pooled_k, _ = pool_sequence_by_similarity(rec["k"].to(dev()), info, matching_results=m)
        assert torch.equal(pooled_k.cpu(), rec["pooled_k_with_q_matching"])
        ref_m = MatchingResults(rec["unpooled_f32"].to(dev()), rec["pooled_f32"].to(dev()))
        y = unpool_sequence_by_similarity(rec["y"].to(dev()), info, ref_m)
        assert torch.equal(y.cpu(), rec["unpooled_seq"])


def test_selection_is_a_partition_at_full_size():
    """Size-independent property at the BASELINE grid (Wan-1.3B, 21x30x52, 12 heads): centres, kept margins and
    dropped margins cover every token exactly once, per head."""
    lat, lw = (21, 30, 52), (3, 3, 2)
    plan = ops.Plan(lat, (3, 10, 4), (3, 3, 3), lw, 0.5)
    g = torch.Generator().manual_seed(5)
    x = torch.randn((1, 12, plan.seq_len, 128), generator=g).to(torch.bfloat16).to(dev())
    un, po, kept, drop = ops.coreset_select(plan, x, want_tokens=True)
    kept, drop = kept.cpu().long(), drop.cpu().long()
    for h in range(12):
        allt = torch.cat([kept[0, h], drop[0, h].flatten()])
        assert torch.equal(allt.sort().values, torch.arange(plan.seq_len))
    # argsort tables are permutations of the margin positions
    both = torch.cat([un, po], dim=-1).cpu().sort(dim=-1).values
    assert torch.equal(both, torch.arange(plan.group_size - 1).expand_as(both))
    # sampled groups agree with the fp64 oracle
    info = O.get_group_info(lat, lw, 0.5)
    un_ref, po_ref = O.match(x[:, :2].cpu().double(), info)
    assert torch.equal(un[:, :2].cpu(), un_ref) and torch.equal(po[:, :2].cpu(), po_ref)


def test_fullsize_index_contract_vs_reference_fp32_and_fp64(golden, capsys):
    """The index contract at the benchmarked geometries (Wan-1.3B 21x30x52, Wan-14B 21x45x80 and the reference's own
    20x45x80), against tables produced by the REFERENCE's pool_sequence_by_similarity run in fp64 and in fp32
    (tests/golden/coreset_fullsize.pt, oracle/make_golden.py):
      * every row of the kernel's tables equals the reference-in-fp64 table;
      * the rows where the kernel differs from the reference-in-fp32 are exactly the rows where the reference's own
        fp32 and fp64 runs differ, and at each of them the fp64 cosine gap between the swapped margins is <= 4e-5
        (what 127 fp32 additions can lose, DESIGN.md section 3.3) — reported below, with counts."""
    from oracle.make_golden import fullsize_coreset_input
    report = []
    for rec in golden("coreset_fullsize.pt"):
        plan = ops.Plan(rec["latent"], (1, 1, 1), (1, 1, 1), rec["window"], rec["rate"])
        assert plan.n_unpooled == rec["n_unpooled"]
        x = fullsize_coreset_input(rec["latent"], rec["heads"], rec["seed"], rec["smooth"]).to(dev())
        un, po = ops.coreset_select(plan, x)
        un8, po8 = un.cpu().to(torch.uint8), po.cpu().to(torch.uint8)
        assert torch.equal(un8, rec["unpooled_f64"]) and torch.equal(po8, rec["pooled_f64"]), rec["name"]
        # reference-in-fp32 tables = fp64 tables with the recorded rows replaced
        order32 = torch.cat([rec["unpooled_f64"], rec["pooled_f64"]], dim=-1)[0].clone()
        at = rec["f32_differs_at"].long()
        order32[at[:, 0], at[:, 1]] = rec["f32_order"]
        mine = torch.cat([un8, po8], dim=-1)[0]
        differs = (mine != order32).any(dim=-1).nonzero()
        assert torch.equal(differs, at), rec["name"]
        gaps = rec["f32_gap"]
        assert gaps.numel() == 0 or gaps.max().item() <= 4e-5, rec["name"]
        report.append(f"{rec['name']}: {rec['n_groups']} (head, group) rows == reference fp64; {at.shape[0]} differ "
                      f"from reference fp32, largest fp64 cosine gap there "
                      f"{(gaps.max().item() if gaps.numel() else 0.0):.2e}")
    with capsys.disabled():
        print("\n[coreset index contract] " + "\n[coreset index contract] ".join(report))


def test_selection_near_ties_and_extreme_magnitudes_match_fp64_oracle():
    """The selection kernel ranks in fp32 and falls back to fp64 when two similarities are closer than the fp32 error
    bound or a norm leaves the range where the bound holds: near-duplicate margins (one bf16 ulp apart in one channel),
    rows scaled by 2^-70 / 2^60 / 2^64 (fp32 squares underflow / stay finite / overflow) and all-zero rows must still
    give the ranking of the fp64 oracle."""
    lat, lw = (8, 6, 8), (2, 3, 2)                      # g = 12, 64 groups
    info = O.get_group_info(lat, lw, 0.5)
    plan = ops.Plan(lat, (1, 1, 1), (1, 1, 1), lw, 0.5)
    g = torch.Generator().manual_seed(11)
    x = torch.randn((1, 3, plan.seq_len, 128), generator=g).to(torch.bfloat16)
    bits = x.view(torch.int16)
    for grp in range(info.margin_indices.shape[0]):
        m = info.margin_indices[grp]
        c = int(info.center_indices[grp, 0])
        # two near-duplicate pairs per group: copy a margin, nudge one channel by one bf16 ulp
        for a, b_, ch in ((0, 1, 5), (4, 7, 100)):
            bits[:, :, m[b_]] = bits[:, :, m[a]]
            bits[:, :, m[b_], ch] += 1
        rows = torch.cat([m, torch.tensor([c])])
        if grp % 8 == 1:
            x[:, :, rows] = (x[:, :, rows].float() * 2.0 ** -70).to(torch.bfloat16)
        elif grp % 8 == 2:
            x[:, :, rows] = (x[:, :, rows].float() * 2.0 ** 60).to(torch.bfloat16)
        elif grp % 8 == 3:
            x[:, :, rows] = (x[:, :, rows].float() * 2.0 ** 64).to(torch.bfloat16)
        elif grp % 8 == 4:
            x[:, :, m[2]] = 0                            # a zero margin row: F.normalize eps path, cos = 0
        elif grp % 8 == 5:
            x[:, :, m[3]] = (x[:, :, m[3]].float() * 2.0 ** -70).to(torch.bfloat16)   # one tiny row among normal ones
    assert torch.isfinite(x.float()).all()
    un, po = ops.coreset_select(plan, x.to(dev()))
    un_ref, po_ref = O.match(x.double(), info)
    assert torch.equal(un.cpu(), un_ref) and torch.equal(po.cpu(), po_ref)


def test_tile_layout_roundtrip_and_reference_order(golden):
    for rec in golden("tile_mask.pt")[:5]:
        lat, tile = rec["latent"], rec["tile"]
        S = lat[0] * lat[1] * lat[2]
        x = FX.det_tensor((1, 2, S, 128), 7).to(torch.bfloat16).to(dev())
        t = tile_layout(x, 1, tile, lat, head_dim=1)
        assert torch.equal(t.cpu(), x.cpu()[:, :, rec["tile_perm"].long()])
        assert torch.equal(untile_layout(t, 1, tile, lat, head_dim=1).cpu(), x.cpu())
        x2 = x.transpose(1, 2).contiguous()                                   # (B, S, H, D) form, head_dim=2
        t2 = tile_layout(x2, 1, tile, lat, head_dim=2)
        assert torch.equal(t2.cpu(), x2.cpu()[:, rec["tile_perm"].long()])


def test_router_scores_and_decisions(golden):
    for rec in golden("router.pt"):
        for dt in (torch.float32, torch.bfloat16):
            w, b, temb = rec["weight"].to(dev(), dt), rec["bias"].to(dev(), dt), rec["temb"].to(dev(), dt)
            bf16 = dt == torch.bfloat16
            ref = O.router_forward(temb.float().cpu(), w.float().cpu(), b.float().cpu(), rec["H"],
                                   module_dtype=torch.bfloat16 if bf16 else None)
            for tau in (None, 0.0, 0.3, 0.36, 0.4, 0.5):
                scores, branch = ops.router_forward(temb, w, b, rec["H"], tau)
                if bf16:
                    # bf16 routers round after SiLU / Linear / Softmax like torch's bf16 modules: bf16-exact scores
                    # within one ulp of the restatement (accumulation order), decisions exact on the kernel's scores
                    got = scores[0].cpu()
                    assert torch.equal(got, got.to(torch.bfloat16).float())
                    assert bool(((got - ref).abs() <= ref.abs() * 2.0 ** -7).all())
                    tau_r = None if tau is None else float(torch.tensor(tau).to(torch.bfloat16))
                    assert torch.equal(branch[0].cpu(), O.route_top1(got, tau_r).to(torch.int32))
                    continue
                assert torch.allclose(scores[0].cpu(), ref, atol=2e-6, rtol=1e-5)
                assert torch.equal(branch[0].cpu(), O.route_top1(ref, tau).to(torch.int32))   # bit-exact decisions
                if dt == torch.float32 and tau is not None:
                    assert torch.equal(branch[0].cpu(), rec["decisions"][tau])                # the reference's own
            if dt == torch.float32:
                assert torch.allclose(scores[0].cpu(), rec["score"], atol=2e-6, rtol=1e-5)


def test_router_module_and_step_routing(golden):
    rec = golden("router.pt")[0]
    routers = []
    for i in range(3):
        r = Router(rec["E"], rec["H"]).to(dev())
        r.load_state_dict({"linear.weight": rec["weight"] * (1 + 0.1 * i), "linear.bias": rec["bias"]})
        routers.append(r)
    temb = rec["temb"].to(dev())
    one = routers[0](temb)
    assert torch.allclose(one.cpu(), rec["score"], atol=2e-6, rtol=1e-5)
    scores, branches = route_step(routers, temb, 0.3)
    assert scores.shape == (3, temb.shape[0], rec["H"], 3) and len(branches) == 3
    for i, r in enumerate(routers):
        ref = O.router_forward(rec["temb"], rec["weight"] * (1 + 0.1 * i), rec["bias"], rec["H"])
        assert branches[i] == O.route_top1(ref, 0.3).tolist()


# ---------------------------------------------------------------------------------------------------------
# attention branches vs the reference's outputs
# ---------------------------------------------------------------------------------------------------------
def _wan_plan():
    c = FX.WAN_CASE
    return ops.Plan(c["latent"], c["tile"], c["window"], c["lowres_window"], c["rate"]), c


def test_wan_branches_vs_reference(golden):
    rec = golden("wan_processor.pt")
    plan, c = _wan_plan()
    q, k, v = (to_dev_bhnd(rec[n]) for n in "qkv")
    H = c["heads"]
    for e, name in ((0, "o_full"), (1, "o_coreset"), (2, "o_sliding")):
        out = ops.routed_attention(plan, q, k, v, branch=[e] * H)
        assert_attn_close(out, rec[name])
    un, po = ops.coreset_select(plan, q)
    assert torch.equal(un.cpu(), rec["unpooled_argsort"]) and torch.equal(po.cpu(), rec["pooled_argsort"])
    # routed mix: head h runs branch h
    out = ops.routed_attention(plan, q, k, v, branch=[0, 1, 2])
    ref = torch.stack([rec["o_full"][:, 0], rec["o_coreset"][:, 1], rec["o_sliding"][:, 2]], dim=1)
    assert_attn_close(out, ref)
    # blended (Train) semantics
    w = torch.tensor(FX.MIX)
    out = ops.routed_attention(plan, q, k, v, weights=w)
    ref = (w[:, :, :, None, None] * torch.stack([rec["o_full"], rec["o_coreset"], rec["o_sliding"]], dim=2)).sum(2)
    assert_attn_close(out, ref)
    # one-hot blend == top-1 routing, exactly (SURVEY.md section 4 invariant 1)
    onehot = torch.tensor([[[1., 0., 0.], [0., 1., 0.], [0., 0., 1.]]])
    a = ops.routed_attention(plan, q, k, v, weights=onehot)
    b = ops.routed_attention(plan, q, k, v, branch=[0, 1, 2])
    assert torch.equal(a, b)


def test_sliding_tile_flex_attn_entry_point(golden):
    rec = golden("wan_processor.pt")
    c = FX.WAN_CASE
    q, k, v = (to_dev_bhnd(rec[n]) for n in "qkv")
    import functools
    sched = create_sliding_tile_attn_mask_func(c["latent"], c["window"], c["tile"], 0, 0)
    fn = functools.partial(lambda *a, **kw: None, block_mask=sched)
    out = sliding_tile_flex_attn(q, k, v, fn, tile_size=c["tile"], latent_shape=c["latent"], head_dim=1)
    assert_attn_close(out, rec["o_sliding"])


def _wan_attn_kwargs(c):
    info = get_group_info(c["latent"], c["lowres_window"], c["rate"], device=dev())
    sched = create_sliding_tile_attn_mask_func(c["latent"], c["window"], c["tile"], 0, 0, dev())
    return dict(lowres_group_info=info, flex_attn_mask_func=sched, window_size=c["window"], tile_size=c["tile"],
                latent_shape=c["latent"])


def _oracle_from_qkv(q, k, v, c, branch=None, weights=None, text_len=0, text_valid=0, kv_from_k=False):
    info = O.get_group_info(c["latent"], c["lowres_window"], c["rate"])
    return O.routed_attention(q.float().cpu(), k.float().cpu(), v.float().cpu(), info, c["latent"], c["window"],
                              c["tile"], branch=branch, weights=weights, text_len=text_len, text_valid=text_valid,
                              kv_from_k=kv_from_k)


def test_wan_processors_vs_reference(golden):
    """Processor-level drop-in: same fake ``attn`` module and hidden states as the reference run.
    (1) the processor's q, k, v against the reference's (bf16 GEMM noise only);
    (2) the processor output against the oracle evaluated on the processor's OWN bf16 q, k, v + fp32 output
        projection — the attention path proper, at the BASELINE tolerance;
    (3) the processor output against the reference's fp32 end-to-end output: bf16 projections and the resulting
        near-tie selection flips (SURVEY.md section 7.3 item 3) bound this one, so the bar is looser."""
    rec = golden("wan_processor.pt")
    c = FX.WAN_CASE
    H = c["heads"]
    S = c["latent"][0] * c["latent"][1] * c["latent"][2]
    attn = FX.FakeWanAttn(H, seed=31).to(dev(), torch.bfloat16)
    attn32 = FX.FakeWanAttn(H, seed=31)
    hs = FX.det_tensor((1, S, H * 128), 32).to(dev(), torch.bfloat16)
    rot = FX.wan_rotary(S, 33).to(dev())
    kw = _wan_attn_kwargs(c)
    mix = torch.tensor(FX.MIX, device=dev())
    ev, tr = WanAttnProcessorTripleEval(check_input=True), WanAttnProcessorTripleTrain(check_input=True)
    q, k, v, _ = ev._input_proj(attn, hs, None, rot)
    for got, name in ((q, "q"), (k, "k"), (v, "v")):
        assert_attn_close(got, rec[name], cos_min=0.9999, max_abs=0.08)

    def out_proj(o):
        with torch.no_grad():
            return attn32.to_out[0](o.transpose(1, 2).flatten(2, 3))

    scale = max(rec["eval_mix"].float().abs().max().item(), 1.0)
    cases = [
        (lambda: ev(attn, hs, None, None, rot, tau_sparse=0.3, routing_score=mix, **kw),
         dict(branch=torch.tensor([0, 1, 2])), "eval_mix"),
        (lambda: ev(attn, hs, None, None, rot, tau_sparse=0.75, routing_score=mix, **kw),
         dict(branch=torch.tensor([0, 1, 0])), "eval_mix_tau075"),       # 0.7 and 0.6 fall below tau -> full
        (lambda: tr(attn, hs, None, None, rot, routing_score=mix, **kw), dict(weights=mix.cpu()), "train_mix"),
    ]
    for run, okw, name in cases:
        with torch.no_grad():
            out = run()
        assert_attn_close(out, out_proj(_oracle_from_qkv(q, k, v, c, **okw)), cos_min=0.999, max_abs=2e-2 * scale)
        assert_attn_close(out, rec[name], cos_min=0.99, max_abs=0.1 * scale)
    out = ev(attn, hs, None, None, rot, tau_sparse=0.3, routing_score=mix, use_original_attn=True, **kw)
    assert_attn_close(out, out_proj(O.full_attention(q.float().cpu(), k.float().cpu(), v.float().cpu())),
                      cos_min=0.999, max_abs=2e-2 * scale)
    assert_attn_close(out, rec["original"], cos_min=0.999, max_abs=3e-2 * scale)
    # reference error behaviour (wan.py:181-193)
    with pytest.raises(ValueError, match="does not match latent shape"):
        ev(attn, hs[:, :-8], None, None, rot, tau_sparse=0.3, routing_score=mix, **kw)
    bad = dict(kw, tile_size=(3, 3, 4))
    with pytest.raises(ValueError, match="does not divide latent shape"):
        ev(attn, hs, None, None, rot, tau_sparse=0.3, routing_score=mix, **bad)


def test_wan_cross_attention_with_i2v_image_keys():
    """Base processor, cross-attention with the I2V image-key branch (wan.py:72-76, 120-139, 154-156): the first 257
    context tokens go through add_k_proj / norm_added_k / add_v_proj, their attention output is added to the text one
    before the output projection.  Reference: the same dataflow in fp32 torch on the same (bf16-valued) weights."""
    import torch.nn as nn
    H, S, T = 2, 200, 40
    attn32 = FX.FakeWanAttn(H, seed=41)
    attn32.add_k_proj, attn32.add_v_proj = nn.Linear(H * 128, H * 128), nn.Linear(H * 128, H * 128)
    attn32.norm_added_k = nn.RMSNorm(H * 128, eps=1e-6)
    FX.fill_module_(attn32, 41)
    attn32 = attn32.to(torch.bfloat16).float()                       # bf16-representable weights on both sides
    attn = FX.FakeWanAttn(H, seed=41)
    attn.add_k_proj, attn.add_v_proj = nn.Linear(H * 128, H * 128), nn.Linear(H * 128, H * 128)
    attn.norm_added_k = nn.RMSNorm(H * 128, eps=1e-6)
    attn.load_state_dict(attn32.state_dict())
    attn = attn.to(dev(), torch.bfloat16)
    hs = FX.det_tensor((1, S, H * 128), 42).to(torch.bfloat16)
    ctx = FX.det_tensor((1, 257 + T, H * 128), 43).to(torch.bfloat16)
    with torch.no_grad():
        out = WanAttnProcessor2_0()(attn, hs.to(dev()), ctx.to(dev()), None, None)
        a, x, c = attn32, hs.float(), ctx.float()
        img, txt = c[:, :257], c[:, 257:]

        def heads(t):
            return t.unflatten(2, (H, -1)).transpose(1, 2)

        q, k, v = heads(a.norm_q(a.to_q(x))), heads(a.norm_k(a.to_k(txt))), heads(a.to_v(txt))
        ki, vi = heads(a.norm_added_k(a.add_k_proj(img))), heads(a.add_v_proj(img))
        o = O.sdpa(q, k, v) + O.sdpa(q, ki, vi)
        ref = a.to_out[0](o.transpose(1, 2).flatten(2, 3))
    assert_attn_close(out, ref, cos_min=0.999, max_abs=2e-2 * max(ref.abs().max().item(), 1.0))


def test_blend_mode_refuses_to_cut_the_router_gradient():
    """The Train blend is how the reference trains its routers (wan.py:296-300).  There is no backward kernel yet:
    asking for one must fail loudly instead of returning a result whose gradient is silently missing."""
    lat, tile, win, lw = (4, 6, 8), (2, 3, 4), (3, 3, 3), (2, 3, 2)
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    g = torch.Generator().manual_seed(3)
    q, k, v = (to_dev_bhnd(torch.randn((1, 2, plan.seq_len, 128), generator=g)) for _ in range(3))
    w = torch.softmax(torch.randn((1, 2, 3), generator=g), -1).to(dev()).requires_grad_(True)
    with pytest.raises(NotImplementedError, match="no backward pass"):
        ops.routed_attention(plan, q, k, v, weights=w)
    with torch.no_grad():
        out = ops.routed_attention(plan, q, k, v, weights=w)
    assert torch.isfinite(out.float()).all()


def _hy_plan():
    c = FX.HUNYUAN_CASE
    return ops.Plan(c["latent"], c["tile"], c["window"], c["lowres_window"], c["rate"], text_len=c["text_len"],
                    text_valid=c["text_valid"]), c


@pytest.mark.parametrize("kind", ["dual", "single"])
def test_hunyuan_branches_vs_reference(golden, kind):
    rec = golden("hunyuan_processor.pt")[kind]
    plan, c = _hy_plan()
    q, k, v = (to_dev_bhnd(rec[n]) for n in "qkv")
    H, S, tv = c["heads"], plan.seq_len, c["text_valid"]
    for e, name in ((0, "o_full"), (1, "o_coreset"), (2, "o_sliding")):
        out = ops.routed_attention(plan, q, k, v, branch=[e] * H, flags=L.ATTN_CORESET_KV_FROM_K)
        assert_attn_close(out, rec[name])
        assert out[:, :, S + tv:].float().abs().max().item() == 0.0      # padded text queries -> exactly zero
    out = ops.routed_attention(plan, q, k, v, branch=[0, 1, 2], flags=L.ATTN_CORESET_KV_FROM_K)
    ref = torch.stack([rec["o_full"][:, 0], rec["o_coreset"][:, 1], rec["o_sliding"][:, 2]], dim=1)
    assert_attn_close(out, ref)


@pytest.mark.parametrize("kind", ["dual", "single"])
def test_hunyuan_processors_vs_reference(golden, kind):
    """Same three-level check as the Wan processor test, for both HunyuanVideo block kinds."""
    rec = golden("hunyuan_processor.pt")[kind]
    c = FX.HUNYUAN_CASE
    S, TL, TV, H = c["latent"][0] * c["latent"][1] * c["latent"][2], c["text_len"], c["text_valid"], c["heads"]
    seed = 42 if kind == "dual" else 43
    attn = FX.FakeHunyuanAttn(H, dual=kind == "dual", seed=seed).to(dev(), torch.bfloat16)
    attn32 = FX.FakeHunyuanAttn(H, dual=kind == "dual", seed=seed)
    hs = FX.det_tensor((1, S, H * 128), 44).to(dev(), torch.bfloat16)
    ehs = FX.det_tensor((1, TL, H * 128), 45).to(dev(), torch.bfloat16)
    mask = torch.zeros(1, 1, 1, S + TL, dtype=torch.bool, device=dev())
    mask[..., :S + TV] = True
    cos_, sin_ = FX.hunyuan_rotary(S, 41)
    rope = (cos_.to(dev()), sin_.to(dev()))
    info = get_group_info(c["latent"], c["lowres_window"], c["rate"], device=dev())
    kw = dict(lowres_group_info=info, flex_attn_mask_func=None, window_size=c["window"], tile_size=c["tile"],
              latent_shape=c["latent"])
    mix = torch.tensor(FX.MIX, device=dev())
    ev = HunyuanVideoFlashAttnProcessorTripleEval(check_input=True)
    tr = HunyuanVideoFlashAttnProcessorTripleTrain(check_input=True)
    with torch.no_grad():       # the forward-only fused prologue, i.e. the q / k / v the Eval processor itself uses
        q, k, v = ev._qkv(attn, hs, ehs, rope)
    for got, name in ((q, "q"), (k, "k"), (v, "v")):
        assert_attn_close(got, rec[name], cos_min=0.9999, max_abs=0.08)

    def out_proj(o):
        with torch.no_grad():
            return ev._step_to_output(attn32, o[:, :, :S], o[:, :, S:])

    scale = max(rec["eval_mix_video"].float().abs().max().item(), 1.0)
    okw = dict(text_len=TL, text_valid=TV, kv_from_k=True)
    a, b = ev(attn, hs, ehs, mask, rope, routing_score=mix, tau_sparse=0.3, **kw)
    ra, rb = out_proj(_oracle_from_qkv(q, k, v, c, branch=torch.tensor([0, 1, 2]), **okw))
    assert_attn_close(a, ra, cos_min=0.999, max_abs=2e-2 * scale)
    assert_attn_close(b, rb, cos_min=0.999, max_abs=2e-2 * scale)
    assert_attn_close(a, rec["eval_mix_video"], cos_min=0.99, max_abs=0.1 * scale)
    assert_attn_close(b, rec["eval_mix_text"], cos_min=0.99, max_abs=0.1 * scale)
    with torch.no_grad():
        a, b = tr(attn, hs, ehs, mask, rope, routing_score=mix, **kw)
    ra, rb = out_proj(_oracle_from_qkv(q, k, v, c, weights=mix.cpu(), **okw))
    assert_attn_close(a, ra, cos_min=0.999, max_abs=2e-2 * scale)
    assert_attn_close(b, rb, cos_min=0.999, max_abs=2e-2 * scale)
    assert_attn_close(a, rec["train_mix_video"], cos_min=0.99, max_abs=0.1 * scale)
    assert_attn_close(b, rec["train_mix_text"], cos_min=0.99, max_abs=0.1 * scale)


# ---------------------------------------------------------------------------------------------------------
# larger seeded cases against the CPU oracle (sizes the oracle finishes in seconds)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lat,tile,win,lw,H,tl,tv", [
    ((10, 12, 16), (5, 6, 4), (3, 3, 3), (2, 3, 2), 4, 0, 0),       # 120-token tiles (reference-native Wan-1.3B tile)
    ((6, 18, 16), (3, 9, 8), (3, 3, 3), (3, 3, 2), 3, 0, 0),        # 216-token tiles, coreset window (3,3,2)
    ((4, 9, 16), (1, 9, 8), (3, 1, 3), (1, 3, 4), 2, 0, 0),         # asymmetric window, coreset window (1,3,4)
    ((6, 12, 8), (3, 6, 4), (3, 3, 3), (2, 3, 2), 3, 40, 23),       # HunyuanVideo-style text tail
    ((2, 4, 8), (1, 2, 4), (5, 5, 5), (2, 2, 2), 2, 8, 8),          # window larger than the grid: degenerates to full
])
def test_branches_vs_oracle(lat, tile, win, lw, H, tl, tv):
    S = lat[0] * lat[1] * lat[2]
    g = torch.Generator().manual_seed(S + H)
    q, k, v = (torch.randn((1, H, S + tl, 128), generator=g).to(torch.bfloat16) for _ in range(3))
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=tl, text_valid=tv)
    info = O.get_group_info(lat, lw, 0.5)
    kv_from_k = tl > 0
    flags = L.ATTN_CORESET_KV_FROM_K if kv_from_k else 0
    qd, kd, vd = to_dev_bhnd(q), to_dev_bhnd(k), to_dev_bhnd(v)
    for e in range(3):
        out = ops.routed_attention(plan, qd, kd, vd, branch=[e] * H, flags=flags)
        ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, win, tile, branch=torch.tensor([e] * H),
                                 text_len=tl, text_valid=tv, kv_from_k=kv_from_k)
        assert_attn_close(out, ref)
    branch = [h % 3 for h in range(H)]
    out = ops.routed_attention(plan, qd, kd, vd, branch=branch, flags=flags)
    ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, win, tile, branch=torch.tensor(branch),
                             text_len=tl, text_valid=tv, kv_from_k=kv_from_k)
    assert_attn_close(out, ref)
    w = torch.softmax(torch.randn((1, H, 3), generator=g), dim=-1)
    out = ops.routed_attention(plan, qd, kd, vd, weights=w, flags=flags)
    ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, win, tile, weights=w, text_len=tl,
                             text_valid=tv, kv_from_k=kv_from_k)
    assert_attn_close(out, ref)


def test_batch_and_head_strides():
    """Batch > 1, head-major (B, H, S, D) memory as well as token-major, and more than one 64-head launch chunk (routed
    and dense)."""
    lat, tile, win, lw = (2, 8, 8), (1, 4, 4), (3, 3, 3), (2, 2, 2)
    S, B, H = 128, 2, 3
    g = torch.Generator().manual_seed(3)
    q, k, v = (torch.randn((B, H, S, 128), generator=g).to(torch.bfloat16) for _ in range(3))
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    info = O.get_group_info(lat, lw, 0.5)
    ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, win, tile, branch=torch.tensor([0, 1, 2]))
    out = ops.routed_attention(plan, q.to(dev()), k.to(dev()), v.to(dev()), branch=[0, 1, 2])     # head-major
    assert_attn_close(out, ref)
    out = ops.routed_attention(plan, to_dev_bhnd(q), to_dev_bhnd(k), to_dev_bhnd(v), branch=[0, 1, 2])
    assert_attn_close(out, ref)
    w = torch.softmax(torch.randn((B, H, 3), generator=g), dim=-1)
    out = ops.routed_attention(plan, q.to(dev()), k.to(dev()), v.to(dev()), weights=w)
    ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, win, tile, weights=w)
    assert_attn_close(out, ref)
    # 72 heads run as launches of 64 + 8 heads; heads are independent, so two calls of 36 heads give the same bits
    H = 72
    q, k, v = (torch.randn((B, S, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2) for _ in range(3))
    out = ops.routed_attention(plan, q, k, v, branch=[0] * H)
    for hs in (slice(0, 36), slice(36, H)):
        assert torch.equal(ops.routed_attention(plan, q[:, hs], k[:, hs], v[:, hs], branch=[0] * 36), out[:, hs])
    q = torch.randn((B, 300, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2)
    k, v = (torch.randn((B, 77, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2) for _ in range(2))
    out = ops.attn_dense(q, k, v)
    for hs in (slice(0, 36), slice(36, H)):
        assert torch.equal(ops.attn_dense(q[:, hs], k[:, hs], v[:, hs]), out[:, hs])


def test_layer_launch_structure():
    """What a layer issues, through the launch and FLOP counters and the per-caller timing: a top-1 layer with every
    branch and a query-half pair (two coreset selections, two pooling gathers, the sliding layout gather, ONE attention
    launch, the zeroing of padded text rows); the same layer blended (one attention launch per branch); 72 full heads and
    72 dense heads (two launches each, at most 64 heads per launch)."""
    def measure(fn):
        torch.cuda.synchronize()
        ops.timing_enable(True)
        ops.timing_collect()
        ops.stats_reset()
        try:
            fn()
            torch.cuda.synchronize()
        finally:
            ops.timing_enable(False)
        kinds = ops.timing_collect_kinds()
        return ops.stats(), kinds["routed"][1:], kinds["dense"][1:]

    g = torch.Generator().manual_seed(23)
    plan = ops.Plan((6, 12, 8), (3, 6, 4), (3, 3, 3), (2, 3, 2), 0.5, text_len=40, text_valid=23)
    S, H = plan.seq_len, 5
    q, k, v = (torch.randn((1, S + 40, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2)
               for _ in range(3))
    w = torch.softmax(torch.randn((1, H, 3), generator=g), -1)
    branch = [0, 1, 2, L.BRANCH_FULL_LO, L.BRANCH_FULL_HI]
    fl = 600639488.0
    assert measure(lambda: ops.routed_attention(plan, q, k, v, branch=branch, flags=L.ATTN_CORESET_KV_FROM_K)) == \
        ((7, fl), (1, fl), (0, 0.0))
    fl = 2084666880.0
    assert measure(lambda: ops.routed_attention(plan, q, k, v, weights=w, flags=L.ATTN_CORESET_KV_FROM_K)) == \
        ((9, fl), (3, fl), (0, 0.0))
    plan = ops.Plan((2, 8, 8), (1, 4, 4), (3, 3, 3), (2, 2, 2), 0.5)
    q, k, v = (torch.randn((2, 72, 128, 128), generator=g).to(torch.bfloat16).to(dev()) for _ in range(3))
    fl = 1207959552.0
    assert measure(lambda: ops.routed_attention(plan, q, k, v, branch=[0] * 72)) == ((2, fl), (2, fl), (0, 0.0))
    q = torch.randn((1, 72, 300, 128), generator=g).to(torch.bfloat16).to(dev())
    k, v = (torch.randn((1, 72, 77, 128), generator=g).to(torch.bfloat16).to(dev()) for _ in range(2))
    fl = 851558400.0
    assert measure(lambda: ops.attn_dense(q, k, v)) == ((2, fl), (0, 0.0), (2, fl))


def test_dense_attention_independent_lengths():
    """Cross-attention shape (wan.py:142-144): 300 queries over 77 / 512 keys."""
    g = torch.Generator().manual_seed(9)
    for nq, nk in ((300, 77), (256, 512), (1, 130)):
        q = torch.randn((2, 3, nq, 128), generator=g).to(torch.bfloat16)
        k = torch.randn((2, 3, nk, 128), generator=g).to(torch.bfloat16)
        v = torch.randn((2, 3, nk, 128), generator=g).to(torch.bfloat16)
        out = ops.attn_dense(to_dev_bhnd(q), to_dev_bhnd(k), to_dev_bhnd(v))
        assert_attn_close(out, O.sdpa(q.float(), k.float(), v.float()))


def _ramp_qkv(n_q, n_k, heads, step, seed):
    """Queries along +-u, keys along u with a magnitude that grows by `step` (natural-log logit units) every 128 keys:
    the row maximum of half of the rows jumps by more than the kernel's lazy-rescale threshold (2^8) at every key block,
    the other half never grows (both cases inside the same warp)."""
    g = torch.Generator().manual_seed(seed)
    u = torch.randn(128, generator=g)
    u = u / u.norm()
    sign = torch.where(torch.arange(n_q) % 3 == 0, -1.0, 1.0)
    q = sign[None, None, :, None] * u * 128 ** 0.5 + 0.05 * torch.randn((1, heads, n_q, 128), generator=g)
    c = step * (torch.arange(n_k) // 128).float()
    k = c[None, None, :, None] * u + 0.05 * torch.randn((1, heads, n_k, 128), generator=g)
    v = torch.randn((1, heads, n_k, 128), generator=g)
    return q.to(torch.bfloat16), k.to(torch.bfloat16), v.to(torch.bfloat16)


def test_lazy_rescale_path_growing_logits():
    """O is rescaled only when a row maximum grows by more than 2^8 after the first block, which random inputs never
    do: force it at every block (the rescale must wait for the PV of the previous block that may still be in flight)."""
    for n_q, n_k, step in ((300, 1100, 8.0), (128, 640, 20.0), (257, 300, 40.0)):
        q, k, v = _ramp_qkv(n_q, n_k, 2, step, seed=n_q)
        out = ops.attn_dense(to_dev_bhnd(q), to_dev_bhnd(k), to_dev_bhnd(v))
        assert_attn_close(out, O.sdpa(q.float(), k.float(), v.float()))


def test_lazy_rescale_path_routed_branches():
    """Same growth through the three branches (run lists, tails, coreset unpool) against the oracle."""
    lat, tile, win, lw = (4, 12, 16), (2, 6, 8), (3, 3, 3), (2, 3, 2)
    S = lat[0] * lat[1] * lat[2]
    q, k, v = _ramp_qkv(S, S, 3, 9.0, seed=21)
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    info = O.get_group_info(lat, lw, 0.5)
    out = ops.routed_attention(plan, to_dev_bhnd(q), to_dev_bhnd(k), to_dev_bhnd(v), branch=[0, 1, 2])
    ref = O.routed_attention(q.float(), k.float(), v.float(), info, lat, win, tile, branch=torch.tensor([0, 1, 2]))
    assert_attn_close(out, ref)


# ---------------------------------------------------------------------------------------------------------
# BASELINE-size properties (size-independent invariants; the oracle is only sampled)
# ---------------------------------------------------------------------------------------------------------
def test_full_size_properties_wan13():
    lat, tile, win, lw, H = (21, 30, 52), (3, 10, 4), (3, 3, 3), (3, 3, 2), 12
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    S = plan.seq_len
    g = torch.Generator().manual_seed(11)
    q, k, v = (torch.randn((1, S, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2) for _ in range(3))
    branch = [h % 3 for h in range(H)]
    out = ops.routed_attention(plan, q, k, v, branch=branch)
    assert torch.isfinite(out.float()).all()
    # (1) softmax rows sum to one in every branch: V = 1 -> O = 1
    ones = torch.ones_like(v)
    o1 = ops.routed_attention(plan, q, k, ones, branch=branch)
    assert (o1.float() - 1).abs().max().item() <= 8e-3
    # (2) linearity in V
    v2 = torch.randn((1, S, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2)
    o2 = ops.routed_attention(plan, q, k, v2, branch=branch)
    osum = ops.routed_attention(plan, q, k, (v.float() + v2.float()).to(torch.bfloat16), branch=branch)
    assert_attn_close(osum, out.float() + o2.float(), max_abs=3e-2)
    # (3) one-hot blend == top-1 routing, exactly
    onehot = torch.nn.functional.one_hot(torch.tensor(branch), 3).float()[None]
    assert torch.equal(ops.routed_attention(plan, q, k, v, weights=onehot), out)
    # (4) sampled rows against the fp32 oracle: a full head, and the window of a few sliding tiles
    qc, kc, vc = q.float().cpu(), k.float().cpu(), v.float().cpu()
    rows = torch.arange(0, S, 257)
    ref = O.sdpa(qc[:, 0:1, rows], kc[:, 0:1], vc[:, 0:1])
    assert_attn_close(out[:, 0:1, rows], ref)
    perm = O.tile_permutation(lat, tile).reshape(-1, plan.tile_tokens)
    wins = O.tile_windows(lat, win, tile)
    nt = [lat[d] // tile[d] for d in range(3)]
    for t in (0, 137, 272):
        lo, hi = wins[t, :3], wins[t, 3:]
        ids = [(a * nt[1] + b) * nt[2] + c for a in range(lo[0], hi[0] + 1) for b in range(lo[1], hi[1] + 1)
               for c in range(lo[2], hi[2] + 1)]
        keys = perm[ids].reshape(-1)
        ref = O.sdpa(qc[:, 2:3, perm[t]], kc[:, 2:3, keys], vc[:, 2:3, keys])
        assert_attn_close(out[:, 2:3, perm[t]], ref)
    # (5) the coreset head against the oracle on its own selection
    info = O.get_group_info(lat, lw, 0.5)
    ref = O.coreset_attention(qc[:, 1:2], kc[:, 1:2], vc[:, 1:2], info)
    assert_attn_close(out[:, 1:2], ref)


def test_full_size_properties_wan14():
    """The headline geometry (BASELINE configs[2]): Wan-14B 720p x 81 f, 21x45x80 = 75,600 tokens, tile (3,9,16) =
    432 tokens (4 query tiles of 128 rows with a 48-row tail, 1296-key runs with a 16-key tail), no text; five heads
    (two full, one coreset, two sliding) so both placements of a branch inside the merged launch are covered."""
    lat, tile, win, lw, H = (21, 45, 80), (3, 9, 16), (3, 3, 3), (3, 3, 2), 5
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    S = plan.seq_len
    assert S == 75600 and plan.tile_tokens == 432 and plan.num_tiles == 175
    g = torch.Generator().manual_seed(17)
    q, k, v = (torch.randn((1, S, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2) for _ in range(3))
    branch = [0, 2, 1, 2, 0]
    out = ops.routed_attention(plan, q, k, v, branch=branch)
    assert torch.isfinite(out.float()).all()
    # (1) softmax rows sum to one in every branch (V = 1 -> O = 1), which also proves every output row was written
    o1 = ops.routed_attention(plan, q, k, torch.ones_like(v), branch=branch)
    assert (o1.float() - 1).abs().max().item() <= 8e-3
    # (2) one-hot blend == top-1 routing, exactly (three separate launches vs the merged one)
    onehot = torch.nn.functional.one_hot(torch.tensor(branch), 3).float()[None]
    assert torch.equal(ops.routed_attention(plan, q, k, v, weights=onehot), out)
    # (3) heads are independent: the same head alone gives the same bits
    for h in (1, 2, 4):
        alone = ops.routed_attention(plan, q[:, h:h + 1], k[:, h:h + 1], v[:, h:h + 1], branch=[branch[h]])
        assert torch.equal(alone, out[:, h:h + 1])
    qc, kc, vc = q.float().cpu(), k.float().cpu(), v.float().cpu()
    # (4) full heads: sampled rows against the fp32 oracle
    rows = torch.arange(0, S, 601)
    for h in (0, 4):
        assert_attn_close(out[:, h:h + 1, rows], O.sdpa(qc[:, h:h + 1, rows], kc[:, h:h + 1], vc[:, h:h + 1]))
    # (5) sliding heads: corner, edge and interior tiles (clamped windows) against the oracle on the window's keys
    perm = O.tile_permutation(lat, tile).reshape(-1, plan.tile_tokens)
    wins = O.tile_windows(lat, win, tile)
    nt = [lat[d] // tile[d] for d in range(3)]
    for h, tiles in ((1, (0, 4, 87, 174)), (3, (12, 90, 170))):
        for t in tiles:
            lo, hi = wins[t, :3], wins[t, 3:]
            ids = [(a * nt[1] + b) * nt[2] + c for a in range(lo[0], hi[0] + 1) for b in range(lo[1], hi[1] + 1)
                   for c in range(lo[2], hi[2] + 1)]
            keys = perm[ids].reshape(-1)
            assert keys.numel() == 27 * 432
            ref = O.sdpa(qc[:, h:h + 1, perm[t]], kc[:, h:h + 1, keys], vc[:, h:h + 1, keys])
            assert_attn_close(out[:, h:h + 1, perm[t]], ref)
    # (6) the coreset head: selection tables equal the fp64 oracle, output equals the oracle on that selection
    info = O.get_group_info(lat, lw, 0.5)
    un, po = ops.coreset_select(plan, q[:, 2:3])
    un_ref, po_ref = O.match(qc[:, 2:3].double(), info)
    assert torch.equal(un.cpu(), un_ref) and torch.equal(po.cpu(), po_ref)
    assert_attn_close(out[:, 2:3], O.coreset_attention(qc[:, 2:3], kc[:, 2:3], vc[:, 2:3], info))


def test_full_size_properties_hunyuan_with_text():
    """HunyuanVideo 720p x 129 f (BASELINE configs[3]): 33x45x80 = 118,800 video tokens + 256 text tokens (64 valid),
    one head per branch (the grid is what matters; 24 heads only repeat it)."""
    lat, tile, win, lw, TL, TV = (33, 45, 80), (3, 9, 16), (3, 3, 3), (3, 3, 2), 256, 64
    plan = ops.Plan(lat, tile, win, lw, 0.5, text_len=TL, text_valid=TV)
    S, H = plan.seq_len, 3
    g = torch.Generator().manual_seed(13)
    q, k, v = (torch.randn((1, S + TL, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2)
               for _ in range(3))
    out = ops.routed_attention(plan, q, k, v, branch=[0, 1, 2], flags=L.ATTN_CORESET_KV_FROM_K)
    assert torch.isfinite(out.float()).all()
    assert out[:, :, S + TV:].float().abs().max().item() == 0.0            # padded text queries -> exactly zero
    ones = torch.ones_like(v)
    o1 = ops.routed_attention(plan, q, k, ones, branch=[0, 1, 2], flags=L.ATTN_CORESET_KV_FROM_K)
    assert (o1[:, :, :S + TV].float() - 1).abs().max().item() <= 8e-3      # softmax rows sum to one everywhere
    qc, kc, vc = q.float().cpu(), k.float().cpu(), v.float().cpu()
    nv = S + TV
    # full head: sampled video rows and every valid text row against the fp32 oracle
    rows = torch.cat([torch.arange(0, S, 1201), torch.arange(S, nv)])
    assert_attn_close(out[:, 0:1, rows], O.sdpa(qc[:, 0:1, rows], kc[:, 0:1, :nv], vc[:, 0:1, :nv]))
    # sliding head: three tiles (window + valid text keys) and the valid text rows (every non-pad key)
    perm = O.tile_permutation(lat, tile).reshape(-1, plan.tile_tokens)
    wins = O.tile_windows(lat, win, tile)
    nt = [lat[d] // tile[d] for d in range(3)]
    text_keys = torch.arange(S, nv)
    for t in (0, 131, 274):
        lo, hi = wins[t, :3], wins[t, 3:]
        ids = [(a * nt[1] + b) * nt[2] + c for a in range(lo[0], hi[0] + 1) for b in range(lo[1], hi[1] + 1)
               for c in range(lo[2], hi[2] + 1)]
        keys = torch.cat([perm[ids].reshape(-1), text_keys])
        assert_attn_close(out[:, 2:3, perm[t]], O.sdpa(qc[:, 2:3, perm[t]], kc[:, 2:3, keys], vc[:, 2:3, keys]))
    assert_attn_close(out[:, 2:3, S:nv], O.sdpa(qc[:, 2:3, S:nv], kc[:, 2:3, :nv], vc[:, 2:3, :nv]))
    # coreset head against the oracle run on the same inputs (K and V pooled with K's matching)
    info = O.get_group_info(lat, lw, 0.5)
    ref = O.coreset_attention(qc[:, 1:2], kc[:, 1:2], vc[:, 1:2], info, TL, TV, kv_from_k=True)
    assert_attn_close(out[:, 1:2], ref)


# ---------------------------------------------------------------------------------------------------------
# Ulysses layout kernels (single GPU: P ranks emulated as one batch of buffers)
# ---------------------------------------------------------------------------------------------------------
def test_ulysses_pack_unpack_kernels():
    from vorta_b200.ulysses import pack_heads, unpack_heads
    P, s_loc, H = 4, 24, 8
    g = torch.Generator().manual_seed(2)
    shards = [torch.randn((1, H, s_loc, 128), generator=g).to(torch.bfloat16) for _ in range(P)]
    want = O.ulysses_scatter_heads(shards)                        # per rank (1, H/P, S, D)
    sends = []
    for r in range(P):
        x = shards[r].transpose(1, 2).reshape(1, s_loc, H, 128).contiguous().to(dev())
        sends.append(pack_heads(x, P)[0])                         # (P, S_loc, hp, D)
    hp = H // P
    for r in range(P):
        recv = torch.stack([sends[p][r] for p in range(P)])       # what the all-to-all delivers to rank r
        got = recv.reshape(P * s_loc, hp, 128).unsqueeze(0).transpose(1, 2)
        assert torch.equal(got.cpu(), want[r])
    # out direction: rank r sends (P, S_loc, hp, D) slices of its (S, hp, D) output; the receiver unpacks
    outs = [w.transpose(1, 2).reshape(P, s_loc, hp, 128).contiguous().to(dev()) for w in want]
    for r in range(P):
        recv = torch.stack([outs[p][r] for p in range(P)])
        y = unpack_heads(recv)                                    # (S_loc, H, D)
        assert torch.equal(y.unsqueeze(0).transpose(1, 2).cpu(), shards[r])


def test_ulysses_pack_unpack_with_balanced_head_table():
    """A slot -> head table only renumbers heads inside the exchange: rank r receives heads head_at[r*hp:(r+1)*hp]
    over the full sequence, and the unpack side returns every head to its own index."""
    from vorta_b200.ulysses import balance_heads, pack_heads, unpack_heads
    P, s_loc, H = 4, 24, 8
    branch = [0, 0, 0, 1, 2, 2, 1, 0]
    head_at = balance_heads(branch, [6.0, 1.6, 1.0], P)
    assert head_at is not None and sorted(head_at) == list(range(H)) and head_at != list(range(H))
    hp = H // P
    g = torch.Generator().manual_seed(3)
    shards = [torch.randn((1, H, s_loc, 128), generator=g).to(torch.bfloat16) for _ in range(P)]
    full = torch.cat(shards, dim=2)                               # (1, H, S, D)
    sends = []
    for r in range(P):
        x = shards[r].transpose(1, 2).reshape(1, s_loc, H, 128).contiguous().to(dev())
        sends.append(pack_heads(x, P, head_at)[0])
    outs = []
    for r in range(P):
        recv = torch.stack([sends[p][r] for p in range(P)])
        got = recv.reshape(P * s_loc, hp, 128).unsqueeze(0).transpose(1, 2)
        assert torch.equal(got.cpu(), full[:, head_at[r * hp:(r + 1) * hp]])
        outs.append(got.transpose(1, 2).reshape(P, s_loc, hp, 128).contiguous())
    for r in range(P):
        recv = torch.stack([outs[p][r] for p in range(P)])
        y = unpack_heads(recv, head_at)
        assert torch.equal(y.unsqueeze(0).transpose(1, 2).cpu(), shards[r])
    with pytest.raises(ValueError):
        pack_heads(x, P, [0] * H)                                 # not a permutation


def test_out_heads_places_local_heads_in_a_wider_output():
    """vb_attn_args.out_heads: a rank holding heads {5, 1, 6} of an 8-head layer writes them at those indices."""
    lat, tile, win, lw = (4, 6, 8), (2, 3, 4), (3, 3, 3), (2, 3, 2)
    S, H_all, mine = 192, 8, [5, 1, 6]
    g = torch.Generator().manual_seed(4)
    q, k, v = (torch.randn((1, H_all, S, 128), generator=g).to(torch.bfloat16).to(dev()) for _ in range(3))
    branch = [0, 1, 2, 0, 1, 2, 0, 1]
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    ref = ops.routed_attention(plan, q, k, v, branch=branch)
    out = torch.zeros((1, S, H_all, 128), dtype=torch.bfloat16, device=dev()).transpose(1, 2)
    ops.routed_attention(plan, q[:, mine], k[:, mine], v[:, mine], branch=[branch[h] for h in mine], out=out,
                         out_heads=mine)
    torch.cuda.synchronize()
    assert torch.equal(out[:, mine], ref[:, mine])
    rest = [h for h in range(H_all) if h not in mine]
    assert out[:, rest].abs().max().item() == 0


def test_bf16_router_matches_reference_router_in_bf16():
    """The reference's inference default is a bf16 router (scripts/wan/inference.py:132).  Its own ``Router`` module
    (vorta/patch/router.py, imported from the staged reference files) run in bf16 on the GPU against the kernel's bf16
    mode: scores within one bf16 ulp (the GEMV accumulation order differs), and the top-1 / threshold decision identical
    for every head whose two best reference scores are more than one ulp apart (closer ones are ties either way)."""
    from oracle import ref_loader
    if not ref_loader.available():
        pytest.skip("reference files not staged (oracle/stage_ref.py)")
    RefRouter = ref_loader.load().router.Router
    torch.manual_seed(7)
    strict = total = 0
    for E, H, B in ((1536, 12, 2), (5120, 40, 1), (3072, 24, 1)):
        ref = RefRouter(E, H, 3).to(dev(), torch.bfloat16)
        mine = Router(E, H).to(dev(), torch.bfloat16)
        mine.load_state_dict(ref.state_dict())
        temb = torch.randn((B, E), device=dev()).to(torch.bfloat16)
        with torch.no_grad():
            want = ref(temb)                                          # (B, H, 3) bf16
        got, _ = ops.router_forward(temb, mine.linear.weight, mine.linear.bias, H)
        got = got[0]
        assert torch.equal(got, got.to(torch.bfloat16).float())      # bf16-exact values in the fp32 buffer
        ulp = want.float().abs() * 2.0 ** -7
        assert bool(((got - want.float()).abs() <= ulp).all())
        for tau in (0.3, 0.36):
            _, branch = ops.router_forward(temb, mine.linear.weight, mine.linear.bias, H, tau)
            s, idx = want[0].topk(1, dim=-1)                          # wan.py:398-400 on the bf16 scores
            idx = idx.clone()
            idx[s < tau] = 0
            top2 = want[0].float().topk(2, dim=-1).values
            clear = ((top2[:, 0] - top2[:, 1]) > 2 * ulp[0].max(dim=-1).values) & \
                    ((top2[:, 0] - tau).abs() > 2 * ulp[0].max(dim=-1).values)
            assert torch.equal(branch[0][clear].cpu(), idx.squeeze(-1)[clear].to(torch.int32).cpu())
            strict += int(clear.sum())
            total += H
    assert strict > 0.5 * total


def test_bf16_router_matches_golden_reference_router_in_bf16(golden):
    """The same bar as above without the reference's files: the weights, inputs and fp32 scores of the reference's own
    ``Router`` (tests/golden/router.pt).  The reference's forward, softmax(linear(silu(temb)).unflatten(1, (H, 3))) in
    plain torch functions (router.py:41-43), first reproduces the reference's fp32 scores, which pins the expression and
    the (head, branch) layout; evaluated in bf16 on the GPU it is then what the reference's module computes in bf16."""
    import torch.nn.functional as F

    def reference_forward(temb, w, b, H):
        return torch.softmax(F.linear(F.silu(temb), w, b).unflatten(1, (H, 3)), dim=-1)

    strict = total = 0
    for rec in golden("router.pt"):
        H = rec["H"]
        assert torch.allclose(reference_forward(rec["temb"], rec["weight"], rec["bias"], H), rec["score"], atol=1e-6)
        w, b, temb = (rec[n].to(dev(), torch.bfloat16) for n in ("weight", "bias", "temb"))
        with torch.no_grad():
            want = reference_forward(temb, w, b, H)                                      # (B, H, 3) bf16
        got = ops.router_forward(temb, w, b, H)[0][0]
        assert torch.equal(got, got.to(torch.bfloat16).float())
        ulp = want.float().abs() * 2.0 ** -7
        assert bool(((got - want.float()).abs() <= ulp).all())
        for tau in (0.3, 0.36):
            _, branch = ops.router_forward(temb, w, b, H, tau)
            s, idx = want[0].topk(1, dim=-1)                                              # wan.py:398-400
            idx = idx.clone()
            idx[s < tau] = 0
            top2 = want[0].float().topk(2, dim=-1).values
            clear = ((top2[:, 0] - top2[:, 1]) > 2 * ulp[0].max(dim=-1).values) & \
                    ((top2[:, 0] - tau).abs() > 2 * ulp[0].max(dim=-1).values)
            assert torch.equal(branch[0][clear].cpu(), idx.squeeze(-1)[clear].to(torch.int32).cpu())
            strict += int(clear.sum())
            total += H
    assert strict > 0.5 * total


def test_query_half_units_equal_the_whole_head():
    """VB_BRANCH_FULL_LO / _HI (Ulysses units finer than a head): the two query halves of a full-attention head, run as
    separate head slots (as two ranks would), write disjoint rows whose union is bit-identical to the whole head;
    mixed with the other branches in one launch; with a HunyuanVideo text tail too."""
    for lat, tile, lw, tl, tv in (((6, 18, 32), (3, 9, 16), (3, 3, 2), 0, 0), ((6, 12, 8), (3, 6, 4), (2, 3, 2), 40, 23)):
        plan = ops.Plan(lat, tile, (3, 3, 3), lw, 0.5, text_len=tl, text_valid=tv)
        S, H = plan.seq_len, 4
        g = torch.Generator().manual_seed(S + 1)
        q, k, v = (torch.randn((1, S + tl, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2)
                   for _ in range(3))
        want = ops.routed_attention(plan, q, k, v, branch=[0, 1, 2, 0])
        # slots: head 0 lower half, head 1 (coreset), head 2 (sliding), head 3 whole, head 0 upper half
        sel = [0, 1, 2, 3, 0]
        qs, ks, vs = (t[:, sel] for t in (q, k, v))
        out = torch.full((1, S + tl, H, 128), float("nan"), dtype=torch.bfloat16, device=dev()).transpose(1, 2)
        ops.routed_attention(plan, qs, ks, vs, branch=[L.BRANCH_FULL_LO, 1, 2, 0, L.BRANCH_FULL_HI], out=out,
                             out_heads=sel)
        torch.cuda.synchronize()
        assert torch.equal(out, want)
        # quarters (VB_BRANCH_FULL_PART(k, 4)) of head 0 in four slots, out of order, next to the whole head 3
        sel = [0, 0, 3, 0, 0]
        ids = [16 + 8 * 4 + 0, 16 + 8 * 4 + 2, 0, 16 + 8 * 4 + 3, 16 + 8 * 4 + 1]
        out4 = torch.full((1, S + tl, H, 128), float("nan"), dtype=torch.bfloat16, device=dev()).transpose(1, 2)
        ops.routed_attention(plan, q[:, sel], k[:, sel], v[:, sel], branch=ids, out=out4, out_heads=sel)
        torch.cuda.synchronize()
        assert torch.equal(out4[:, [0, 3]], want[:, [0, 3]])
        with pytest.raises(L.VortaB200Error):            # more kinds of parts than a launch has segments for
            six = [16 + 8 * 4 + i for i in range(4)] + [L.BRANCH_FULL_LO, L.BRANCH_FULL_HI]
            ops.routed_attention(plan, q[:, [0] * 6], k[:, [0] * 6], v[:, [0] * 6], branch=six)
        with pytest.raises(ValueError):                  # part 4 of 4 does not exist
            ops.routed_attention(plan, q[:, :1], k[:, :1], v[:, :1], branch=[16 + 8 * 4 + 4])
        # one half alone leaves the other half's rows untouched
        out2 = torch.zeros_like(out)
        ops.routed_attention(plan, qs[:, :1], ks[:, :1], vs[:, :1], branch=[L.BRANCH_FULL_LO], out=out2, out_heads=[0])
        torch.cuda.synchronize()
        written = out2[0, 0].float().abs().sum(dim=-1) > 0
        assert 0 < int(written.sum()) < S + tv
        assert torch.equal(out2[0, 0][written], want[0, 0][written])


def test_ulysses_scatter_with_placement_table():
    """vb_ulysses_scatter_qkv_slots on one GPU, the P ranks' receive buffers emulated as P local buffers: every unit of
    the placement (uneven head counts, a head sent to two ranks) lands in its slot over the full sequence."""
    import ctypes as C
    P, s_loc, H, slots = 4, 24, 8, 4
    placement = [[(0, 1), (5, 0)], [(0, 2), (1, 0), (2, 0)], [(3, 0), (4, 0), (6, 0), (7, 0)], []]
    g = torch.Generator().manual_seed(9)
    shards = [[torch.randn((1, s_loc, H, 128), generator=g).to(torch.bfloat16).to(dev()).transpose(1, 2)
               for _ in range(3)] for _ in range(P)]
    S = P * s_loc
    bufs = [torch.zeros((3, S, slots, 128), dtype=torch.bfloat16, device=dev()) for _ in range(P)]
    ptrs = (C.c_void_p * P)(*[b.data_ptr() for b in bufs])
    peers, sl, hd = [], [], []
    for p, units in enumerate(placement):
        for slot, (h, _) in enumerate(units):
            peers.append(p); sl.append(slot); hd.append(h)
    arr = C.c_int32 * len(peers)
    i64x3 = C.c_int64 * 3
    for r in range(P):
        q, k, v = shards[r]
        L.check(L.lib().vb_ulysses_scatter_qkv_slots(
            q.data_ptr(), k.data_ptr(), v.data_ptr(), i64x3(q.stride(2), k.stride(2), v.stride(2)),
            i64x3(q.stride(1), k.stride(1), v.stride(1)), ptrs, S, s_loc, slots, P, r, arr(*peers), arr(*sl), arr(*hd),
            len(peers), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    full = [torch.cat([shards[r][t] for r in range(P)], dim=2) for t in range(3)]          # (1, H, S, 128)
    for p, units in enumerate(placement):
        for slot, (h, _) in enumerate(units):
            for t in range(3):
                assert torch.equal(bufs[p][t, :, slot], full[t][0, h])
        assert bufs[p][:, :, len(units):].abs().max().item() == 0 if len(units) < slots else True
