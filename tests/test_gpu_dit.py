"""DiT-level drop-in tests: the patched Wan / HunyuanVideo shells (fused block kernels + routed attention + one-launch
routing) against a plain PyTorch fp32 restatement of the reference's block dataflow
(vorta/patch/modeling_wan.py:38-239) with the oracle's attention."""
import pytest
import torch
import torch.nn.functional as F

from oracle import vorta_oracle as O
from vorta_b200.dit import HunyuanConfig, HunyuanDiT, WanDiT
from vorta_b200.dit import wan as wan_mod
from vorta_b200.patch import apply_vorta_transformer, modeling_hunyuan, prepare_hunyuan_self_attn_kwargs
from vorta_b200.patch import prepare_wan_self_attn_kwargs

pytestmark = pytest.mark.gpu

LAT, TILE, WIN, LW = (4, 6, 8), (2, 3, 4), (3, 3, 3), (2, 3, 2)


def _wan_reference_forward(model, latents, timestep, text, branches, info):
    """fp32 CPU restatement of wan_transformer_3d_routed_forward / wan_block_routed_forward."""
    m = model
    cfg = m.config
    H = cfg.heads
    x = m.patch_embedding(latents).flatten(2).transpose(1, 2)
    temb, tproj, ctx, _ = m.condition_embedder(timestep, text)
    tproj = tproj.unflatten(1, (6, -1))
    rot = m.rope(latents)                                                   # (1, 1, S, 64) complex128

    def rope(t):                                                           # wan.py:34-37
        z = torch.view_as_complex(t.double().unflatten(3, (-1, 2)))
        return torch.view_as_real(z * rot).flatten(3, 4).float()

    def heads(t):
        return t.unflatten(2, (H, -1)).transpose(1, 2)

    for li, blk in enumerate(m.blocks):
        sh, sc, g, csh, csc, cg = (blk.scale_shift_table + tproj.float()).chunk(6, dim=1)
        n = F.layer_norm(x, (cfg.dim,), None, None, cfg.eps) * (1 + sc) + sh
        a = blk.attn1
        q, k, v = a.norm_q(a.to_q(n)), a.norm_k(a.to_k(n)), a.to_v(n)
        q, k, v = rope(heads(q)), rope(heads(k)), heads(v)
        o = O.routed_attention(q, k, v, info, LAT, WIN, TILE, branch=torch.tensor(branches[li]))
        x = x + a.to_out[0](o.transpose(1, 2).flatten(2, 3)) * g
        n = F.layer_norm(x, (cfg.dim,), blk.norm2.weight, blk.norm2.bias, cfg.eps)
        a = blk.attn2
        q, k, v = heads(a.norm_q(a.to_q(n))), heads(a.norm_k(a.to_k(ctx))), heads(a.to_v(ctx))
        x = x + a.to_out[0](O.sdpa(q, k, v).transpose(1, 2).flatten(2, 3))
        n = F.layer_norm(x, (cfg.dim,), None, None, cfg.eps) * (1 + csc) + csh
        x = x + blk.ffn.proj_out(F.gelu(blk.ffn.proj_in(n), approximate="tanh")) * cg
    shift, scale = (m.scale_shift_table + temb.unsqueeze(1)).chunk(2, dim=1)
    x = F.layer_norm(x, (cfg.dim,), None, None, cfg.eps) * (1 + scale) + shift
    x = m.proj_out(x)
    B = latents.shape[0]
    x = x.reshape(B, LAT[0], LAT[1], LAT[2], 1, 2, 2, -1).permute(0, 7, 1, 4, 2, 5, 3, 6)
    return x.flatten(6, 7).flatten(4, 5).flatten(2, 3)


def test_wan_dit_step_matches_torch_reference():
    _wan_dit_step_check(dim=384, heads=3)


def test_wan_dit_step_at_a_production_width():
    """dim 1536 (Wan-1.3B): the block kernels run their warp-per-row instances inside a whole step (at 384 channels
    every row kernel takes the CTA-per-row fallback)."""
    _wan_dit_step_check(dim=1536, heads=12)


def _wan_dit_step_check(dim, heads):
    wan_mod.WAN_CONFIGS["tiny"] = wan_mod.WanConfig(dim=dim, heads=heads, ffn_dim=512, num_layers=3, text_dim=64)
    dev = torch.device("cuda:0")
    model = WanDiT.build("tiny", dev, torch.bfloat16, seed=3)
    apply_vorta_transformer(model, router_dtype=torch.float32)
    kw = prepare_wan_self_attn_kwargs(dict(latent_shape=LAT, window_size=WIN, tile_size=TILE, lowres_window_size=LW,
                                           lowres_reduction_rate=0.5), dev, tau_sparse=0.3)
    g = torch.Generator().manual_seed(4)
    latents = torch.randn((1, 16, LAT[0], 2 * LAT[1], 2 * LAT[2]), generator=g)
    text = torch.randn((1, 20, 64), generator=g)
    ts = torch.tensor([431.0])
    # make the routers decisive and varied so that every branch appears
    with torch.no_grad():
        for li, blk in enumerate(model.blocks):
            pattern = torch.tensor([[3., 0., 0.], [0., 3., 0.], [0., 0., 3.]]).roll(li, 0)
            blk.router.linear.bias.copy_(pattern[torch.arange(heads) % 3].flatten())
    with torch.no_grad():
        res = model(latents.to(dev, torch.bfloat16), ts.to(dev), text.to(dev, torch.bfloat16),
                    self_attention_kwargs=kw, return_routing_scores=True)
    out, scores = res.sample, res.routing_scores                    # RoutedTransformerModelOutput (outputs.py:8-14)
    assert res.reg_loss is None and res[0] is out and len(res.to_tuple()) == 2
    branches = [s[0].float().argmax(-1).tolist() for s in scores]
    assert sorted(set(sum(branches, []))) == [0, 1, 2]
    # reference: same weights (bf16 values) in fp32 on the CPU
    ref_model = WanDiT.build("tiny", "cpu", torch.float32, seed=3)
    apply_vorta_transformer(ref_model)                                     # same module tree / state-dict keys
    ref_model.load_state_dict({k: v.float().cpu() for k, v in model.state_dict().items()})
    info = O.get_group_info(LAT, LW, 0.5)
    with torch.no_grad():
        ref = _wan_reference_forward(ref_model, latents.bfloat16().float(), ts, text.bfloat16().float(), branches, info)
    assert out.shape == ref.shape == latents.shape
    o, r = out.float().cpu(), ref
    cos = F.cosine_similarity(o.flatten(), r.flatten(), dim=0).item()
    assert torch.isfinite(o).all() and cos >= 0.995, cos
    assert (o - r).abs().max().item() <= 0.08 * max(r.abs().max().item(), 1.0)


def test_hunyuan_dit_step_runs_and_respects_routing():
    """HunyuanVideo shell: a step runs through dual- and single-stream blocks with routed joint attention; forcing every
    head to the full branch must equal the unrouted (use_original_attn) processors."""
    dev = torch.device("cuda:0")
    cfg = HunyuanConfig(heads=3, num_layers=2, num_single_layers=2, text_embed_dim=64, pooled_projection_dim=32)
    model = HunyuanDiT.build(cfg, dev, torch.bfloat16, seed=5)
    modeling_hunyuan.apply_vorta_transformer(model, router_dtype=torch.float32)
    lat, tile, win, lw = (2, 8, 8), (1, 4, 4), (3, 3, 3), (2, 2, 2)
    kw = prepare_hunyuan_self_attn_kwargs(dict(latent_shape=lat, window_size=win, tile_size=tile,
                                               lowres_window_size=lw, lowres_reduction_rate=0.5), dev, tau_sparse=0.3)
    g = torch.Generator().manual_seed(6)
    x = torch.randn((1, 16, lat[0], 2 * lat[1], 2 * lat[2]), generator=g).to(dev, torch.bfloat16)
    text = torch.randn((1, 16, 64), generator=g).to(dev, torch.bfloat16)
    mask = torch.zeros((1, 16), dtype=torch.bool, device=dev)
    mask[:, :11] = True
    pooled = torch.randn((1, 32), generator=g).to(dev, torch.bfloat16)
    ts, guidance = torch.tensor([500.0], device=dev), torch.tensor([6000.0], device=dev)
    blocks = list(model.transformer_blocks) + list(model.single_transformer_blocks)

    def run(bias):
        with torch.no_grad():
            for blk in blocks:
                blk.router.linear.weight.zero_()
                blk.router.linear.bias.copy_(torch.tensor(bias).flatten())
            res = model(x, ts, text, mask, pooled, guidance, self_attention_kwargs=dict(kw),
                        return_routing_scores=True, return_dict=False)
            assert len(res) == 5 and res[1] is None and res[2] is None and res[3] is None      # reference 5-tuple
            return res[0], res[4]

    out_mix, scores = run([[4., 0., 0.], [0., 4., 0.], [0., 0., 4.]])
    assert out_mix.shape == x.shape and torch.isfinite(out_mix.float()).all()
    assert [s[0].float().argmax(-1).tolist() for s in scores] == [[0, 1, 2]] * 4
    out_full, _ = run([[4., 0., 0.]] * 3)
    # unrouted processors on the same weights
    modeling_hunyuan.apply_sp_flashattn_transformer(model)
    orig = {}
    for blk in blocks:          # block forwards pass routing kwargs; the baseline processor ignores routing
        orig[blk] = blk.attn.processor
    with torch.no_grad():
        for blk in blocks:
            blk.attn.set_processor(_Unrouted(blk.attn.processor))
        out_plain = model(x, ts, text, mask, pooled, guidance, self_attention_kwargs=dict(kw)).sample
    assert torch.equal(out_full, out_plain)
    assert not torch.equal(out_mix, out_full)


class _Unrouted:
    """Adapter: call the baseline HunyuanVideo processor, dropping the routing kwargs the routed block forward adds."""

    def __init__(self, proc):
        self.proc = proc

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, image_rotary_emb=None,
                 **_):
        return self.proc(attn, hidden_states, encoder_hidden_states, attention_mask, image_rotary_emb)


def test_wan_denoise_loop_cfg_and_routing_scores():
    """Denoising loop of wan_pipeline_call (pipeline_wan.py:323-365) on the tiny shell: equals a hand-written loop of
    the same forwards; guidance_scale <= 1 makes a single forward per step; routing scores come back per step."""
    from vorta_b200.patch.pipeline import FlowMatchEulerScheduler, wan_denoise
    wan_mod.WAN_CONFIGS["tiny"] = wan_mod.WanConfig(dim=384, heads=3, ffn_dim=512, num_layers=2, text_dim=64)
    dev = torch.device("cuda:0")
    model = WanDiT.build("tiny", dev, torch.bfloat16, seed=7)
    apply_vorta_transformer(model, router_dtype=torch.float32)
    kw = prepare_wan_self_attn_kwargs(dict(latent_shape=LAT, window_size=WIN, tile_size=TILE, lowres_window_size=LW,
                                           lowres_reduction_rate=0.5), dev, tau_sparse=0.3)
    g = torch.Generator().manual_seed(8)
    noise = torch.randn((1, 16, LAT[0], 2 * LAT[1], 2 * LAT[2]), generator=g).to(dev)
    pos = torch.randn((1, 20, 64), generator=g).to(dev)
    neg = torch.randn((1, 20, 64), generator=g).to(dev)
    steps, scale = 3, 5.0
    out = wan_denoise(model, FlowMatchEulerScheduler(shift=3.0), noise.clone(), pos, neg, guidance_scale=scale,
                      num_inference_steps=steps, self_attention_kwargs=kw, return_routing_scores=True)
    assert out.frames.shape == noise.shape and out.frames.dtype == torch.float32
    assert len(out.routing_scores) == steps and len(out.routing_scores[0]) == 2
    assert tuple(out.routing_scores[0][0].shape) == (1, 3, 3)
    # hand-written loop
    sch = FlowMatchEulerScheduler(shift=3.0)
    sch.set_timesteps(steps, device=dev)
    x = noise.clone()
    calls = 0
    with torch.no_grad():
        for i, t in enumerate(sch.timesteps):
            xin, ts = x.to(torch.bfloat16), t.expand(1)
            c = model(xin, ts, pos.to(torch.bfloat16), self_attention_kwargs=kw)[0]
            u = model(xin, ts, neg.to(torch.bfloat16), self_attention_kwargs=kw, return_dict=False)[0]
            calls += 2
            v = u + scale * (c - u)
            x = (x.float() + (sch.sigmas[i + 1] - sch.sigmas[i]) * v.float())
    assert torch.equal(out.frames, x)
    assert float(sch.sigmas[-1]) == 0.0 and abs(float(sch.sigmas[0]) - 1.0) < 1e-6
    # no CFG: one forward per step and a different trajectory
    lat2, _ = wan_denoise(model, FlowMatchEulerScheduler(shift=3.0), noise.clone(), pos, neg, guidance_scale=1.0,
                          num_inference_steps=steps, self_attention_kwargs=kw, return_dict=False)
    assert lat2.shape == noise.shape and not torch.equal(lat2, out.frames)


def test_hunyuan_denoise_loop_runs():
    from vorta_b200.patch.pipeline import FlowMatchEulerScheduler, hunyuan_denoise
    dev = torch.device("cuda:0")
    cfg = HunyuanConfig(heads=3, num_layers=1, num_single_layers=1, text_embed_dim=64, pooled_projection_dim=32)
    model = HunyuanDiT.build(cfg, dev, torch.bfloat16, seed=9)
    modeling_hunyuan.apply_vorta_transformer(model, router_dtype=torch.float32)
    lat, tile, win, lw = (2, 8, 8), (1, 4, 4), (3, 3, 3), (2, 2, 2)
    kw = prepare_hunyuan_self_attn_kwargs(dict(latent_shape=lat, window_size=win, tile_size=tile,
                                               lowres_window_size=lw, lowres_reduction_rate=0.5), dev, tau_sparse=0.3)
    g = torch.Generator().manual_seed(10)
    noise = torch.randn((1, 16, lat[0], 2 * lat[1], 2 * lat[2]), generator=g).to(dev)
    text = torch.randn((1, 16, 64), generator=g).to(dev)
    mask = torch.zeros((1, 16), dtype=torch.bool, device=dev)
    mask[:, :9] = True
    pooled = torch.randn((1, 32), generator=g).to(dev)
    before = kw.get("flex_attn_mask_func")
    out = hunyuan_denoise(model, FlowMatchEulerScheduler(shift=7.0), noise.clone(), text, mask, pooled,
                          guidance_scale=6.0, num_inference_steps=2, self_attention_kwargs=kw,
                          return_routing_scores=True)
    assert out.frames.shape == noise.shape and torch.isfinite(out.frames).all()
    assert len(out.routing_scores) == 2 and len(out.routing_scores[0]) == 2
    assert kw.get("flex_attn_mask_func") is before        # the caller's kwargs are not mutated (deep copy, :378)


def test_wan_forward_reference_return_structure_and_losses():
    """Return structure of wan_transformer_3d_routed_forward (modeling_wan.py:174-186) and the router-training
    losses in the forward direction (:109-171) with the Train processors: L2 on the full-attention score summed over
    blocks, hidden / last layer distillation against the un-routed blocks."""
    wan_mod.WAN_CONFIGS["tiny"] = wan_mod.WanConfig(dim=384, heads=3, ffn_dim=512, num_layers=2, text_dim=64)
    dev = torch.device("cuda:0")
    model = WanDiT.build("tiny", dev, torch.bfloat16, seed=11)
    apply_vorta_transformer(model, train_router=True, router_dtype=torch.float32)
    kw = prepare_wan_self_attn_kwargs(dict(latent_shape=LAT, window_size=WIN, tile_size=TILE, lowres_window_size=LW,
                                           lowres_reduction_rate=0.5), dev)
    g = torch.Generator().manual_seed(12)
    x = torch.randn((1, 16, LAT[0], 2 * LAT[1], 2 * LAT[2]), generator=g).to(dev, torch.bfloat16)
    text = torch.randn((1, 20, 64), generator=g).to(dev, torch.bfloat16)
    ts = torch.tensor([431.0], device=dev)
    with torch.no_grad():
        res = model(x, ts, text, self_attention_kwargs=kw, return_losses=True, reture_hidden_layer_distill_loss=True,
                    return_routing_scores=True)
        tup = model(x, ts, text, self_attention_kwargs=kw, return_dict=False)
    assert len(tup) == 5 and tup[1] is None and tup[2] is None and tup[3] is None and tup[4] == []
    assert torch.equal(tup[0], res.sample)
    want_reg = sum(torch.square(s[:, :, 0].float()).mean() for s in res.routing_scores)
    assert abs(float(res.reg_loss) - float(want_reg)) < 2e-3 * float(want_reg)      # squared in the router's bf16 output dtype
    assert float(res.last_layer_distill_loss) > 0 and float(res.hidden_layer_distill_loss) > 0
    assert all(s.device.type == "cpu" and tuple(s.shape) == (1, 3, 3) for s in res.routing_scores)
    # training through the blend is refused loudly (no attention backward yet)
    with pytest.raises(NotImplementedError):
        model(x, ts, text, self_attention_kwargs=kw)


def test_wan_dense_baseline_forward_equals_all_full_routing():
    """apply_sp_flashattn_transformer (modeling_wan.py:313-323): the un-routed baseline runs through the same
    token-sharded forward with the base processors; it must equal the routed model when every head is routed to the full
    branch (same kernel, same q / k / v), and refuse router outputs."""
    from vorta_b200.patch import apply_sp_flashattn_transformer
    wan_mod.WAN_CONFIGS["tiny"] = wan_mod.WanConfig(dim=384, heads=3, ffn_dim=512, num_layers=2, text_dim=64)
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(6)
    latents = torch.randn((1, 16, LAT[0], 2 * LAT[1], 2 * LAT[2]), generator=g).to(dev, torch.bfloat16)
    text = torch.randn((1, 20, 64), generator=g).to(dev, torch.bfloat16)
    ts = torch.tensor([431.0], device=dev)
    routed = WanDiT.build("tiny", dev, torch.bfloat16, seed=8)
    apply_vorta_transformer(routed, router_dtype=torch.float32)
    with torch.no_grad():
        for blk in routed.blocks:
            blk.router.linear.weight.zero_()
            blk.router.linear.bias.copy_(torch.tensor([4., 0., 0.]).repeat(3))      # every head -> full attention
    kw = prepare_wan_self_attn_kwargs(dict(latent_shape=LAT, window_size=WIN, tile_size=TILE, lowres_window_size=LW,
                                           lowres_reduction_rate=0.5), dev, tau_sparse=0.3)
    with torch.no_grad():
        want = routed(latents, ts, text, self_attention_kwargs=kw, return_dict=False)[0]
    dense = WanDiT.build("tiny", dev, torch.bfloat16, seed=8)
    apply_sp_flashattn_transformer(dense)
    with torch.no_grad():
        got = dense(latents, ts, text, return_dict=False)[0]
        assert torch.equal(got, want)
        with pytest.raises(ValueError):
            dense(latents, ts, text, return_routing_scores=True)
