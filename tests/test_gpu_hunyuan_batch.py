"""HunyuanVideo at batch > 1: every sample has its own un-padded text length.

Contract: output sample b of a batch call is bit-identical to a batch-1 call on sample b alone with a plan whose
text_valid is that sample's length, for every branch mix, top-1 and blend modes, CORESET_KV_FROM_K and the dense
(use_original_attn) path; rows [S + tv[b], S + text_len) of sample b are exactly 0.  Above the attention call (projection
GEMMs, whose algorithm cuBLAS may pick by the number of rows) the bar is bf16 tolerance: |got - ref| <= 0.02 + 0.02 |ref|,
three times that for the denoise loop with true CFG at scale 2.
"""
import pytest
import torch

from oracle import fixtures as FX
from vorta_b200 import _lib as L
from vorta_b200 import ops

pytestmark = pytest.mark.gpu

LAT, TILE, WIN, LW, TL = (6, 12, 8), (3, 6, 4), (3, 3, 3), (2, 3, 2), 40
S = LAT[0] * LAT[1] * LAT[2]
N = S + TL
H = 6
PLAN_TV = 23                                  # the plan's own length: sample 0 of the first case runs its tables
LENGTHS = {"distinct": [23, 40, 0], "two-equal": [7, 40, 7]}
FP = L.branch_full_part
BRANCHES = {
    "full": [0] * H,
    "coreset": [1] * H,
    "sliding": [2] * H,
    "mixed": [2, 0, 1, 1, 2, 0],
    "query-parts": [FP(0, 2), FP(1, 2), 1, FP(0, 3), FP(2, 3), 2],
}
SENTINEL = 0x7FA1          # a bf16 NaN: no attention output has these bits
GUARD = 3


def dev():
    L.check(L.lib().vb_device_check())
    return torch.device("cuda:0")


def plan_of(tv):
    return ops.Plan(LAT, TILE, WIN, LW, 0.5, text_len=TL, text_valid=tv)


def qkv(B, seed):
    """(B, H, N, 128) bf16 views over (B, N, H, 128) memory; the padded text rows hold data too (they must be ignored)."""
    g = torch.Generator().manual_seed(seed)
    return [torch.randn((B, N, H, 128), generator=g).to(dev(), torch.bfloat16).transpose(1, 2) for _ in range(3)]


def fenced(B, H_out):
    """A sentinel-filled buffer and the (B, H_out, N, 128) output view inside it: guard rows, a head on either side."""
    buf = torch.full((B, N + 2 * GUARD, H_out + 2, 128), SENTINEL, dtype=torch.int16, device=dev())
    return buf, buf.view(torch.bfloat16)[:, GUARD:GUARD + N, 1:1 + H_out].transpose(1, 2)


def run_fenced(plan, q, k, v, tvs, branch=None, weights=None, flags=0):
    buf, out = fenced(q.shape[0], H)
    ops.routed_attention(plan, q, k, v, branch=branch, weights=weights, flags=flags, out=out, text_valid=tvs)
    torch.cuda.synchronize()
    return buf, out


def closed_form_flops(tvs, branch=None, blend=False):
    """Sum over samples of the per-head closed forms of BASELINE.md section 3, each with the sample's own length."""
    total = 0.0
    for tv in tvs:
        p = plan_of(tv)
        if blend:
            total += H * sum(p.flops_per_head(e) for e in range(3))
        else:
            total += sum(p.flops_per_head(e) for e in branch)
    return total


def check_against_batch1(tvs, branch=None, weights=None, flags=0, seed=1):
    """The batch call vs one batch-1 call per sample: the whole fenced buffers must be equal (so the batch call writes
    exactly the rows the batch-1 calls write, and the same bits), padded rows zero."""
    B = len(tvs)
    q, k, v = qkv(B, seed)
    plan = plan_of(PLAN_TV)
    ops.stats_reset()
    buf, out = run_fenced(plan, q, k, v, tvs, branch=branch, weights=weights, flags=flags)
    _, flops = ops.stats()
    for b, tv in enumerate(tvs):
        ref_buf, _ = run_fenced(plan_of(tv), q[b:b + 1], k[b:b + 1], v[b:b + 1], None, branch=branch,
                                weights=None if weights is None else weights[b:b + 1], flags=flags)
        assert torch.equal(buf[b:b + 1], ref_buf), f"sample {b} (text_valid {tv}) differs from its batch-1 call"
        # heads that own padded rows: whole heads, and the last query part of a split head
        writes_pad = [h for h in range(H)
                      if branch is None or branch[h] < 16 or (branch[h] - 16) % 8 == (branch[h] - 16) // 8 - 1]
        assert torch.count_nonzero(out[b, writes_pad, S + tv:].float()) == 0, f"padded rows of sample {b} not zero"
    return flops


@pytest.mark.parametrize("lengths", list(LENGTHS), ids=list(LENGTHS))
@pytest.mark.parametrize("mix", list(BRANCHES), ids=list(BRANCHES))
@pytest.mark.parametrize("flags", [0, L.ATTN_CORESET_KV_FROM_K], ids=["kv-own", "kv-from-k"])
def test_top1_batch_equals_batch1_per_sample(lengths, mix, flags):
    tvs, branch = LENGTHS[lengths], BRANCHES[mix]
    flops = check_against_batch1(tvs, branch=branch, flags=flags, seed=3)
    if mix != "query-parts":
        assert flops == pytest.approx(closed_form_flops(tvs, branch), rel=1e-9)


@pytest.mark.parametrize("lengths", list(LENGTHS), ids=list(LENGTHS))
@pytest.mark.parametrize("flags", [0, L.ATTN_CORESET_KV_FROM_K], ids=["kv-own", "kv-from-k"])
def test_blend_batch_equals_batch1_per_sample(lengths, flags):
    tvs = LENGTHS[lengths]
    g = torch.Generator().manual_seed(5)
    weights = torch.softmax(torch.randn((len(tvs), H, 3), generator=g) * 2, -1).to(dev())
    flops = check_against_batch1(tvs, weights=weights, flags=flags, seed=4)
    assert flops == pytest.approx(closed_form_flops(tvs, blend=True), rel=1e-9)


def test_fence_and_padded_rows_explicit():
    """Every row of every head is written (the padded ones as 0), nothing outside the output view is."""
    tvs = LENGTHS["distinct"]
    q, k, v = qkv(3, 7)
    buf, out = run_fenced(plan_of(PLAN_TV), q, k, v, tvs, branch=BRANCHES["mixed"])
    mask = torch.zeros(buf.shape[:3], dtype=torch.bool, device=buf.device)
    mask[:, GUARD:GUARD + N, 1:1 + H] = True
    assert not bool(((buf != SENTINEL).any(dim=-1) & ~mask).any()), "a row outside the output view was written"
    assert bool((buf[:, GUARD:GUARD + N, 1:1 + H] != SENTINEL).any(dim=-1).all()), "an output row was not written"
    for b, tv in enumerate(tvs):
        assert torch.count_nonzero(out[b, :, S + tv:].float()) == 0
        if tv:
            assert torch.count_nonzero(out[b, :, S + tv - 1].float()) > 0


def test_more_length_groups_than_one_grid_holds():
    """Nine samples of nine lengths: 9 x 3 segments split over several grids, each sample still bit-exact."""
    tvs = [40, 0, 23, 1, 39, 17, 8, 31, 2]
    check_against_batch1(tvs, branch=BRANCHES["mixed"], flags=L.ATTN_CORESET_KV_FROM_K, seed=8)


def test_cached_lengths_stay_bounded_and_correct():
    """More distinct lengths over successive calls than the plan caches: older schedules are dropped and rebuilt, the
    results do not change."""
    plan = plan_of(PLAN_TV)
    q, k, v = qkv(2, 9)
    first = None
    for rnd in range(2):
        outs = []
        for tv in range(0, TL + 1, 2):
            outs.append(ops.routed_attention(plan, q, k, v, branch=BRANCHES["mixed"], text_valid=[tv, TL - tv]).clone())
        if first is None:
            first = outs
        else:
            assert all(torch.equal(a, b) for a, b in zip(first, outs))


def test_text_valid_errors():
    plan = plan_of(PLAN_TV)
    q, k, v = qkv(3, 10)
    with pytest.raises(ValueError):
        ops.routed_attention(plan, q, k, v, branch=BRANCHES["mixed"], text_valid=[23, TL + 1, 0])
    with pytest.raises(ValueError):
        ops.routed_attention(plan, q, k, v, branch=BRANCHES["mixed"], text_valid=[23, -1, 0])
    with pytest.raises(ValueError):
        ops.routed_attention(plan, q, k, v, branch=BRANCHES["mixed"], text_valid=[23, 40])


# ---------------------------------------------------------------------------------------------------------
# processors, blocks, DiT and denoise loop
# ---------------------------------------------------------------------------------------------------------
P_LAT, P_TILE, P_WIN, P_LW, P_TL = (2, 8, 8), (1, 4, 4), (3, 3, 3), (2, 2, 2), 16
P_S, P_H = 128, 4
P_TV = [11, 5]


def close(got, ref, what="", amplify=1.0):
    """|got - ref| <= amplify * (0.02 + 0.02 |ref|): bf16 tolerance, times the factor by which the caller's arithmetic
    can magnify a rounding difference of one forward."""
    got, ref = got.float(), ref.float()
    bad = (got - ref).abs() > amplify * (0.02 + 0.02 * ref.abs())
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} elements beyond bf16 tolerance, max err " \
                                f"{(got - ref).abs().max().item():.3e}"


def _processor_inputs(dual):
    from vorta_b200.attention import get_group_info
    d = dev()
    attn = FX.FakeHunyuanAttn(P_H, dual=dual, seed=11).to(d, torch.bfloat16)
    hs = FX.det_tensor((2, P_S, P_H * 128), 12).to(d, torch.bfloat16)
    ehs = FX.det_tensor((2, P_TL, P_H * 128), 13).to(d, torch.bfloat16)
    mask = torch.zeros(2, 1, 1, P_S + P_TL, dtype=torch.bool, device=d)
    for b, tv in enumerate(P_TV):
        mask[b, ..., :P_S + tv] = True
    c, s = FX.hunyuan_rotary(P_S, 14)
    kw = dict(lowres_group_info=get_group_info(P_LAT, P_LW, 0.5, device=d), flex_attn_mask_func=None,
              window_size=P_WIN, tile_size=P_TILE, latent_shape=P_LAT)
    score = torch.softmax(FX.det_tensor((2, P_H, 3), 8, 4.0), -1).to(d)
    return attn, hs, ehs, mask, (c.to(d), s.to(d)), kw, score


def _processors():
    from vorta_b200.attention import (HunyuanVideoFlashAttnProcessor, HunyuanVideoFlashAttnProcessorTripleEval,
                                      HunyuanVideoFlashAttnProcessorTripleTrain)
    return {
        "dense": (HunyuanVideoFlashAttnProcessor(), lambda kw, sc: {}),
        "eval": (HunyuanVideoFlashAttnProcessorTripleEval(), lambda kw, sc: dict(kw, routing_score=sc, tau_sparse=0.3)),
        "train": (HunyuanVideoFlashAttnProcessorTripleTrain(), lambda kw, sc: dict(kw, routing_score=sc)),
        "train-original": (HunyuanVideoFlashAttnProcessorTripleTrain(),
                           lambda kw, sc: dict(kw, routing_score=sc, use_original_attn=True)),
    }


@pytest.mark.parametrize("dual", [True, False], ids=["dual-stream", "single-stream"])
@pytest.mark.parametrize("name", ["dense", "eval", "train", "train-original"])
def test_processor_attention_bitwise_and_output_within_tolerance(dual, name):
    """B = 2 with different masks through the processor: the attention output (same Q / K / V) equals the per-sample
    calls bitwise; the full processor output (with its projections) matches within bf16 tolerance.  Eval routing comes
    from sample 0's scores for the batch, so the per-sample reference uses sample 0's scores too."""
    attn, hs, ehs, mask, rope, kw, score = _processor_inputs(dual)
    proc, extra = _processors()[name]
    with torch.no_grad():
        full_v, full_t = proc(attn, hs, ehs, mask, rope, **extra(kw, score))
        qkv_all = proc._qkv(attn, hs, ehs, rope)
        proc._qkv = lambda *a: qkv_all
        proc._step_to_output = lambda attn_, v, t: (v, t)           # the attention output itself
        att_v, att_t = proc(attn, hs, ehs, mask, rope, **extra(kw, score))
        for b in range(2):
            sc = score[b:b + 1] if name.startswith("train") else score[:1]
            proc._qkv = lambda *a, b=b: tuple(t[b:b + 1] for t in qkv_all)
            ref_v, ref_t = proc(attn, hs[b:b + 1], ehs[b:b + 1], mask[b:b + 1], rope, **extra(kw, sc))
            assert torch.equal(att_v[b:b + 1], ref_v) and torch.equal(att_t[b:b + 1], ref_t), f"sample {b}"
            assert torch.count_nonzero(att_t[b, :, P_TV[b]:].float()) == 0
            del proc._qkv, proc._step_to_output
            one_v, one_t = proc(attn, hs[b:b + 1], ehs[b:b + 1], mask[b:b + 1], rope, **extra(kw, sc))
            close(full_v[b:b + 1], one_v, f"video output of sample {b}")
            close(full_t[b:b + 1], one_t, f"text output of sample {b}")
            proc._qkv = lambda *a: qkv_all
            proc._step_to_output = lambda attn_, v, t: (v, t)


def _dit_setup(seed):
    from vorta_b200.dit import HunyuanConfig, HunyuanDiT
    from vorta_b200.patch import modeling_hunyuan, prepare_hunyuan_self_attn_kwargs
    d = dev()
    cfg = HunyuanConfig(heads=3, num_layers=2, num_single_layers=2, text_embed_dim=64, pooled_projection_dim=32)
    model = HunyuanDiT.build(cfg, d, torch.bfloat16, seed=seed)
    modeling_hunyuan.apply_vorta_transformer(model, router_dtype=torch.float32)
    kw = prepare_hunyuan_self_attn_kwargs(dict(latent_shape=P_LAT, window_size=P_WIN, tile_size=P_TILE,
                                               lowres_window_size=P_LW, lowres_reduction_rate=0.5), d, tau_sparse=0.3)
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn((2, 16, P_LAT[0], 2 * P_LAT[1], 2 * P_LAT[2]), generator=g).to(d)
    text = torch.randn((2, 16, 64), generator=g).to(d)
    mask = torch.zeros((2, 16), dtype=torch.bool, device=d)
    for b, tv in enumerate(P_TV):
        mask[b, :tv] = True
    pooled = torch.randn((2, 32), generator=g).to(d)
    blocks = list(model.transformer_blocks) + list(model.single_transformer_blocks)
    with torch.no_grad():          # routing that uses every branch in every layer
        for blk in blocks:
            blk.router.linear.weight.zero_()
            blk.router.linear.bias.copy_(torch.tensor([[4., 0., 0.], [0., 4., 0.], [0., 0., 4.]]).flatten())
    return model, kw, x, text, mask, pooled


def test_hunyuan_dit_batch2_matches_per_sample():
    model, kw, x, text, mask, pooled = _dit_setup(21)
    d = x.device
    x = x.to(torch.bfloat16)
    text, pooled = text.to(torch.bfloat16), pooled.to(torch.bfloat16)
    ts, guidance = torch.tensor([500.0, 500.0], device=d), torch.tensor([6000.0, 6000.0], device=d)
    with torch.no_grad():
        out = model(x, ts, text, mask, pooled, guidance, self_attention_kwargs=dict(kw), return_dict=False)[0]
        for b in range(2):
            one = model(x[b:b + 1], ts[:1], text[b:b + 1], mask[b:b + 1], pooled[b:b + 1], guidance[:1],
                        self_attention_kwargs=dict(kw), return_dict=False)[0]
            close(out[b:b + 1], one, f"DiT sample {b}")


def test_hunyuan_denoise_batch2_matches_per_sample():
    """True CFG forms neg + s (pred - neg): a rounding difference of either forward reaches the update magnified by up to
    |s| + |1 - s| = 3 at s = 2, so the bar is three times the bf16 tolerance."""
    from vorta_b200.patch.pipeline import FlowMatchEulerScheduler, hunyuan_denoise
    model, kw, noise, text, mask, pooled = _dit_setup(31)
    neg_text = torch.randn_like(text)
    neg_mask = mask.flip(0)
    run = lambda sl: hunyuan_denoise(model, FlowMatchEulerScheduler(shift=7.0), noise[sl].clone(), text[sl], mask[sl],
                                     pooled[sl], guidance_scale=6.0, num_inference_steps=2, self_attention_kwargs=kw,
                                     negative_prompt_embeds=neg_text[sl], negative_prompt_attention_mask=neg_mask[sl],
                                     negative_pooled_prompt_embeds=pooled[sl], true_cfg_scale=2.0).frames
    out = run(slice(0, 2))
    assert out.shape == noise.shape and torch.isfinite(out).all()
    for b in range(2):
        close(out[b:b + 1], run(slice(b, b + 1)), f"denoised sample {b}", amplify=3.0)
