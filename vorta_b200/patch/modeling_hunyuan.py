"""Install boundary for HunyuanVideo — the reference's ``vorta/patch/modeling_hunyuan.py`` (apply_vorta_transformer
:648-706, hunyuan_transformer_3d_routed_forward :165-449, hunyuan_single_block_routed_forward :452-521,
hunyuan_dual_block_routed_forward :524-590, hunyuan_rope_forward :593-618, hunyuan_combined_embedding_forward :621-645).

Same design deltas as ``modeling_wan.py``: one router launch per step (the routers read the clean timestep embedding
only, :491/:555/:645), token sharding under Ulysses (text tokens replicated), fused elementwise passes, training
losses in the forward direction only.  The per-prompt sliding-tile schedule needs no BlockMask rebuild (:232-241): the valid text length is a field
of the plan.
"""
from __future__ import annotations

import os
from typing import Any, Dict, Optional, Tuple

import torch
import torch.nn.functional as F

from .. import ops
from ..attention import (HunyuanVideoFlashAttnProcessor, HunyuanVideoFlashAttnProcessorTripleEval,
                         HunyuanVideoFlashAttnProcessorTripleTrain)
from ..ulysses import SP_STATE, all_gather
from .modeling_wan import accumulate_loss, load_router_checkpoint
from .outputs import RoutedTransformerModelOutput
from .router import Router, route_step


def _rotary_1d(dim: int, pos: torch.Tensor, theta: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """cos / sin (N, dim), pair-repeated — the ``use_real=True`` layout of diffusers' get_1d_rotary_pos_embed that
    hunyuan_rope_forward calls (:611-613)."""
    freqs = 1.0 / (theta ** (torch.arange(0, dim, 2, dtype=torch.float32, device=pos.device)[: dim // 2] / dim))
    ang = torch.outer(pos.float(), freqs)
    return ang.cos().repeat_interleave(2, dim=1), ang.sin().repeat_interleave(2, dim=1)


def hunyuan_rope_forward(self, hidden_states: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(cos, sin), each (T*H*W, 128), for the FULL token grid (:593-618); processors narrow it per rank."""
    _, _, num_frames, height, width = hidden_states.shape
    sizes = [num_frames // self.patch_size_t, height // self.patch_size, width // self.patch_size]
    grids = torch.meshgrid(*[torch.arange(0, s, device=hidden_states.device, dtype=torch.float32) for s in sizes],
                           indexing="ij")
    parts = [_rotary_1d(self.rope_dim[i], grids[i].reshape(-1), self.theta) for i in range(3)]
    return torch.cat([p[0] for p in parts], dim=1), torch.cat([p[1] for p in parts], dim=1)


def hunyuan_combined_embedding_forward(self, timestep, pooled_projection, guidance=None):
    """conditioning, token_replace_emb, clean timestep embedding (the routers' input) (:621-645)."""
    dtype = pooled_projection.dtype
    timesteps_emb = self.timestep_embedder(self.time_proj(timestep).to(dtype))
    conditioning = timesteps_emb + self.text_embedder(pooled_projection)
    if self.guidance_embedder is not None and guidance is not None:
        conditioning = conditioning + self.guidance_embedder(self.time_proj(guidance).to(dtype))
    return conditioning, None, timesteps_emb


def _ada_chunks(norm, emb: torch.Tensor, n: int):
    """The n fp32 modulation vectors of an adaptive LayerNorm module, through the members diffusers' AdaLayerNormZero
    (6), AdaLayerNormZeroSingle (3) and AdaLayerNormContinuous (2: scale, shift) all have — ``silu`` and ``linear`` — so
    the fused block forwards work on the diffusers model as well as on ``vorta_b200.dit.HunyuanDiT``; the LayerNorm
    itself is applied by ``ops.ln_modulate`` (reference call sites: modeling_hunyuan.py:146, 471, 538-539)."""
    return norm.linear(norm.silu(emb)).float().chunk(n, dim=1)


def _attn_kwargs(self_attention_kwargs, routing_score, branch):
    kw = dict(self_attention_kwargs or {})
    kw["routing_score"] = routing_score
    if branch is not None:
        kw["branch"] = branch
    return kw


def _text_valid_kw(self_attention_kwargs):
    """{"text_valid": [n_0, ...]} when the transformer forward counted every prompt's un-padded tokens once for the
    whole step."""
    tv = (self_attention_kwargs or {}).get("text_valid")
    return {} if tv is None else {"text_valid": tv}


def hunyuan_dual_block_routed_forward(self, hidden_states, encoder_hidden_states, temb, attention_mask, freqs_cis,
                                      token_replace_emb=None, first_frame_num_tokens: int = 0,
                                      use_original_attn: bool = False, self_attention_kwargs=None,
                                      clean_timesteps_emb=None, routing_score=None, branch=None):
    """Dataflow of :524-590 with every elementwise stage as one fused pass."""
    shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = _ada_chunks(self.norm1, temb, 6)
    c_shift_msa, c_scale_msa, c_gate_msa, c_shift_mlp, c_scale_mlp, c_gate_mlp = _ada_chunks(self.norm1_context, temb, 6)
    norm_hidden = ops.ln_modulate(hidden_states, None, None, scale_msa, shift_msa, 1e-6)
    norm_encoder = ops.ln_modulate(encoder_hidden_states, None, None, c_scale_msa, c_shift_msa, 1e-6)
    if use_original_attn:
        attn_out, ctx_out = self.attn(hidden_states=norm_hidden, encoder_hidden_states=norm_encoder,
                                      attention_mask=attention_mask, image_rotary_emb=freqs_cis, use_original_attn=True,
                                      **_text_valid_kw(self_attention_kwargs))
    else:
        if routing_score is None:
            routing_score = self.router(clean_timesteps_emb)
        attn_out, ctx_out = self.attn(hidden_states=norm_hidden, encoder_hidden_states=norm_encoder,
                                      attention_mask=attention_mask, image_rotary_emb=freqs_cis,
                                      **_attn_kwargs(self_attention_kwargs, routing_score, branch))
    hidden_states = ops.gate_residual(hidden_states, attn_out, gate_msa)
    encoder_hidden_states = ops.gate_residual(encoder_hidden_states, ctx_out, c_gate_msa)
    ff = self.ff(ops.ln_modulate(hidden_states, None, None, scale_mlp, shift_mlp, 1e-6))
    ff_ctx = self.ff_context(ops.ln_modulate(encoder_hidden_states, None, None, c_scale_mlp, c_shift_mlp, 1e-6))
    hidden_states = ops.gate_residual(hidden_states, ff, gate_mlp)
    encoder_hidden_states = ops.gate_residual(encoder_hidden_states, ff_ctx, c_gate_mlp)
    return hidden_states, encoder_hidden_states, routing_score


def hunyuan_single_block_routed_forward(self, hidden_states, encoder_hidden_states, temb, attention_mask,
                                        image_rotary_emb, token_replace_emb=None, first_frame_num_tokens: int = 0,
                                        use_original_attn: bool = False, self_attention_kwargs=None,
                                        clean_timesteps_emb=None, routing_score=None, branch=None):
    """Dataflow of :452-521."""
    text_len = encoder_hidden_states.shape[1]
    residual = torch.cat([hidden_states, encoder_hidden_states], dim=1)
    shift, scale, gate = _ada_chunks(self.norm, temb, 3)
    norm = ops.ln_modulate(residual, None, None, scale, shift, 1e-6)
    mlp = torch._addmm_activation(self.proj_mlp.bias, norm.flatten(0, 1), self.proj_mlp.weight.t(),
                                  use_gelu=True).unflatten(0, norm.shape[:2])
    norm_hidden, norm_encoder = norm[:, :-text_len], norm[:, -text_len:]
    if use_original_attn:
        attn_out, ctx_out = self.attn(hidden_states=norm_hidden, encoder_hidden_states=norm_encoder,
                                      attention_mask=attention_mask, image_rotary_emb=image_rotary_emb,
                                      use_original_attn=True, **_text_valid_kw(self_attention_kwargs))
    else:
        if routing_score is None:
            routing_score = self.router(clean_timesteps_emb)
        attn_out, ctx_out = self.attn(hidden_states=norm_hidden, encoder_hidden_states=norm_encoder,
                                      attention_mask=attention_mask, image_rotary_emb=image_rotary_emb,
                                      **_attn_kwargs(self_attention_kwargs, routing_score, branch))
    attn = torch.cat([attn_out, ctx_out], dim=1)
    out = self.proj_out(torch.cat([attn, mlp], dim=2))
    out = ops.gate_residual(residual, out, gate)
    return out[:, :-text_len], out[:, -text_len:], routing_score


def hunyuan_transformer_3d_routed_forward(self, hidden_states: torch.Tensor, timestep: torch.Tensor,
                                          encoder_hidden_states: torch.Tensor, encoder_attention_mask: torch.Tensor,
                                          pooled_projections: torch.Tensor, guidance: Optional[torch.Tensor] = None,
                                          attention_kwargs=None, return_dict: bool = True,
                                          self_attention_kwargs: Optional[Dict[str, Any]] = None,
                                          return_losses: bool = False, reture_hidden_layer_distill_loss: bool = False,
                                          return_routing_scores: bool = False):
    """One DiT forward = one denoise step: signature, dataflow and return structure of :165-449
    (``return_dict=False`` -> ``(sample, reg_loss, last_layer_distill_loss, hidden_layer_distill_loss,
    routing_scores)``); ``return_losses`` evaluates the router-training losses in the forward direction only."""
    batch_size, _, num_frames, height, width = hidden_states.shape
    p, p_t = self.config.patch_size, self.config.patch_size_t
    ppf, pph, ppw = num_frames // p_t, height // p, width // p

    image_rotary_emb = self.rope(hidden_states)
    temb, token_replace_emb, clean_emb = self.time_text_embed(timestep, pooled_projections, guidance)
    hidden_states = self.x_embedder(hidden_states).flatten(2).transpose(1, 2).contiguous()
    encoder_hidden_states = self.context_embedder(encoder_hidden_states, timestep, encoder_attention_mask)   # :210

    latent_len, text_len = hidden_states.shape[1], encoder_hidden_states.shape[1]
    if SP_STATE.enabled:        # token sharding of the video stream; the text stream is replicated
        s_loc = latent_len // SP_STATE.sp_size
        hidden_states = hidden_states.narrow(1, SP_STATE.group_local_rank * s_loc, s_loc).contiguous()
    attention_mask = torch.zeros(batch_size, latent_len + text_len, device=hidden_states.device, dtype=torch.bool)
    effective = latent_len + encoder_attention_mask.sum(dim=1, dtype=torch.int)             # :213-229
    for i in range(batch_size):
        attention_mask[i, : effective[i]] = True
    attention_mask = attention_mask.unsqueeze(1).unsqueeze(1)

    kwargs = dict(self_attention_kwargs or {})
    tau = kwargs.get("tau_sparse")
    # the un-padded text length of every sample, ONE host read per step instead of one per layer (hunyuan.py:169 syncs
    # in every block)
    kwargs["text_valid"] = [int(e) - latent_len for e in effective.tolist()]
    blocks = list(self.transformer_blocks) + list(self.single_transformer_blocks)
    eval_mode = isinstance(blocks[0].attn.processor, HunyuanVideoFlashAttnProcessorTripleEval)
    if not eval_mode and torch.is_grad_enabled() and any(q.requires_grad for q in blocks[0].router.parameters()):
        # the Train processors exist to fit the routers; that needs the backward of the attention kernels
        raise NotImplementedError("vorta_b200: router training is not supported yet (no attention backward); run the "
                                  "Train processors under torch.no_grad()")
    scores, branches = route_step([b.router for b in blocks], clean_emb, tau if eval_mode else None)
    self._vb_last_branches = branches if eval_mode else None      # fp32 decisions of this step, per layer (bench / tests)
    reg_loss = hidden_layer_distill_loss = last_layer_distill_loss = None
    ref_hidden_states = hidden_states.detach().clone() if return_losses else None
    ref_encoder_hidden_states = encoder_hidden_states.detach().clone() if return_losses else None
    for i, block in enumerate(blocks):
        score_i = scores[i].to(temb.dtype)
        hidden_states, encoder_hidden_states, _ = block(
            hidden_states, encoder_hidden_states, temb, attention_mask, image_rotary_emb, token_replace_emb, 0,
            use_original_attn=False, self_attention_kwargs=kwargs, clean_timesteps_emb=clean_emb,
            routing_score=score_i, branch=branches[i] if eval_mode else None)
        if return_losses:
            with torch.no_grad():                          # reference branch: the un-routed block (:357-368)
                ref_hidden_states, ref_encoder_hidden_states, _ = block(
                    ref_hidden_states, ref_encoder_hidden_states, temb, attention_mask, image_rotary_emb,
                    token_replace_emb, 0, use_original_attn=True, self_attention_kwargs=_text_valid_kw(kwargs))
            reg_loss = accumulate_loss(reg_loss, torch.square(score_i[:, :, 0]).mean().float())
            if reture_hidden_layer_distill_loss:
                hidden_layer_distill_loss = accumulate_loss(
                    hidden_layer_distill_loss, F.mse_loss(ref_hidden_states.float(), hidden_states.float()))
    routing_scores = list(scores.detach().to(temb.dtype).cpu().unbind(0)) if return_routing_scores else []

    scale, shift = _ada_chunks(self.norm_out, temb, 2)
    hidden_states = self.proj_out(ops.ln_modulate(hidden_states, None, None, scale, shift, 1e-6))
    if return_losses:
        with torch.no_grad():
            ref_hidden_states = self.proj_out(ops.ln_modulate(ref_hidden_states, None, None, scale, shift, 1e-6))
        last_layer_distill_loss = F.mse_loss(ref_hidden_states.float(), hidden_states.float())
    if SP_STATE.enabled:
        hidden_states = all_gather(hidden_states, dim=1)
    hidden_states = hidden_states.reshape(batch_size, ppf, pph, ppw, -1, p_t, p, p)
    hidden_states = hidden_states.permute(0, 4, 1, 5, 2, 6, 3, 7)
    output = hidden_states.flatten(6, 7).flatten(4, 5).flatten(2, 3)
    if not return_dict:
        return (output, reg_loss, last_layer_distill_loss, hidden_layer_distill_loss, routing_scores)
    return RoutedTransformerModelOutput(sample=output, reg_loss=reg_loss, last_layer_distill_loss=last_layer_distill_loss,
                                        hidden_layer_distill_loss=hidden_layer_distill_loss,
                                        routing_scores=routing_scores)


def apply_vorta_transformer(model, train_router: bool = False, checkpoint_file: Optional[os.PathLike] = None,
                            attn_processor_kwargs: Optional[Dict[str, Any]] = None,
                            router_dtype: Optional[torch.dtype] = None):
    """Same signature and effect as modeling_hunyuan.py:648-706."""
    cls = HunyuanVideoFlashAttnProcessorTripleTrain if train_router else HunyuanVideoFlashAttnProcessorTripleEval
    model.__class__.forward = hunyuan_transformer_3d_routed_forward
    model.rope.__class__.forward = hunyuan_rope_forward
    model.time_text_embed.__class__.forward = hunyuan_combined_embedding_forward
    param = next(model.parameters())
    dtype = router_dtype or param.dtype
    kw = dict(attn_processor_kwargs or {})
    kw.update(check_input=True)
    for block in model.transformer_blocks:
        if not hasattr(block, "router"):
            block.router = Router(block.norm1.linear.in_features, block.attn.heads).to(device=param.device, dtype=dtype)
        if train_router:
            block.router.requires_grad_(True)
        block.attn.set_processor(cls(**kw))
        kw.update(check_input=False)                      # only the first block checks (:685)
        block.__class__.forward = hunyuan_dual_block_routed_forward
    for block in model.single_transformer_blocks:
        if not hasattr(block, "router"):
            block.router = Router(block.norm.linear.in_features, block.attn.heads).to(device=param.device, dtype=dtype)
        if train_router:
            block.router.requires_grad_(True)
        block.attn.set_processor(cls(**kw))
        block.__class__.forward = hunyuan_single_block_routed_forward
    if checkpoint_file is not None:
        load_router_checkpoint(checkpoint_file, model)
    return model


def apply_sp_flashattn_transformer(model):
    """Baseline-only variant (:709-723)."""
    model.rope.__class__.forward = hunyuan_rope_forward
    for block in list(model.transformer_blocks) + list(model.single_transformer_blocks):
        block.attn.set_processor(HunyuanVideoFlashAttnProcessor())
    return model
