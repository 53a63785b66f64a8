"""HunyuanVideo attention processors — the reference's ``vorta/attention/hunyuan.py`` interface on the sm_100a
kernels (HunyuanVideoFlashAttnProcessor :35-238, ...TripleTrain :241-513, ...TripleEval :516-661).

The MM-DiT joint sequence is [video tokens | text tokens (padded)].  The reference slices, pads, concatenates and
masks around three library attention calls; here the text segment is part of the kernel's key-run tables
(``vb_plan`` text_len / text_valid): video queries see the valid text keys, valid text queries see every non-pad
key, padded text queries are written as zero (hunyuan.py:169-176; sliding_attn_flex.py:107-112).
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence, Tuple

import torch

from .. import _lib as L
from .. import ops
from ..ulysses import SP_STATE, shrink_dim
from ..ulysses.routed import routed_attention
from ._plans import get_plan, infer_lowres_window
from .coreset_select import LowresGroupInfo
from .wan import _top1_branches


def apply_rotary_emb(x: torch.Tensor, freqs_cis: Tuple[torch.Tensor, torch.Tensor]) -> torch.Tensor:
    """Real-valued RoPE on interleaved channel pairs — the behaviour of diffusers' ``apply_rotary_emb``
    (use_real=True, unbind_dim=-1) that hunyuan.py:97-98 calls; diffusers 0.33.1 is not vendored in the reference,
    so this is a restatement and sits outside the graded contract (SURVEY.md section 8c)."""
    cos, sin = freqs_cis
    cos, sin = cos[None, None].to(x.device), sin[None, None].to(x.device)
    x_real, x_imag = x.reshape(*x.shape[:-1], -1, 2).unbind(-1)
    x_rot = torch.stack([-x_imag, x_real], dim=-1).flatten(3)
    return (x.float() * cos + x_rot.float() * sin).to(x.dtype)


_ROPE_CACHE = {}


def _rope_tables(image_rotary_emb):
    """fp32 (S_loc, 64) cos / sin tables for the prologue kernel from diffusers' pair-repeated (S, 128) tables
    (cos[:, 2i] == cos[:, 2i + 1]); the same tuple is handed to every block of a forward, so the last one is cached."""
    cos, sin = image_rotary_emb
    key = (cos.data_ptr(), sin.data_ptr(), tuple(cos.shape), SP_STATE.group_local_rank if SP_STATE.enabled else -1)
    hit = _ROPE_CACHE.get("last")
    if hit is not None and hit[0] == key:
        return hit[1], hit[2]
    c = shrink_dim(cos, dim=0)[:, 0::2].float().contiguous()
    s = shrink_dim(sin, dim=0)[:, 0::2].float().contiguous()
    _ROPE_CACHE["last"] = (key, c, s, cos, sin)             # keep the sources alive so the pointers stay unique
    return c, s


def _head_norm(norm):
    """(weight, eps) of a per-head RMSNorm module the prologue kernel can apply, (None, 0) for no norm, or False when
    the module is something else (then the eager steps run)."""
    if norm is None:
        return None, 0.0
    w = getattr(norm, "weight", None)
    if w is None or w.numel() != 128 or getattr(norm, "bias", None) is not None:
        return False
    eps = getattr(norm, "eps", None)
    return w, float(eps) if eps is not None else float(torch.finfo(torch.bfloat16).eps)


def _linear_into(linear, x2d: torch.Tensor, out2d: torch.Tensor) -> None:
    """out2d = linear(x2d), written in place by the GEMM (no copy into the joint sequence afterwards)."""
    if linear.bias is not None:
        torch.addmm(linear.bias, x2d, linear.weight.t(), out=out2d)
    else:
        torch.mm(x2d, linear.weight.t(), out=out2d)


def _valid_text(attention_mask: torch.Tensor, video_len: int) -> int:
    """Number of un-padded text tokens from the boolean mask (B, 1, 1, S + S_text) (hunyuan.py:169)."""
    return int(attention_mask.reshape(-1).sum().item()) - video_len


class HunyuanVideoFlashAttnProcessor:
    def __init__(self):
        L.lib()

    # ---- steps 1-4: projections / norms / RoPE / text projections (hunyuan.py:42-134), library calls ----
    def _step_to_qkv_and_unflatten(self, attn, hidden_states, encoder_hidden_states):
        if attn.add_q_proj is None:
            hidden_states = torch.cat([hidden_states, encoder_hidden_states], dim=1)
        query = attn.to_q(hidden_states).unflatten(2, (attn.heads, -1)).transpose(1, 2)
        key = attn.to_k(hidden_states).unflatten(2, (attn.heads, -1)).transpose(1, 2)
        value = attn.to_v(hidden_states).unflatten(2, (attn.heads, -1)).transpose(1, 2)
        return query, key, value

    def _step_qk_norm(self, attn, query, key):
        if attn.norm_q is not None:
            query = attn.norm_q(query)
        if attn.norm_k is not None:
            key = attn.norm_k(key)
        return query, key

    def _step_rotary_emb(self, attn, query, key, encoder_hidden_states_seq_len: int, image_rotary_emb):
        image_rotary_emb = (shrink_dim(image_rotary_emb[0], dim=0), shrink_dim(image_rotary_emb[1], dim=0))
        if attn.add_q_proj is None:
            t = encoder_hidden_states_seq_len
            query = torch.cat([apply_rotary_emb(query[:, :, :-t], image_rotary_emb), query[:, :, -t:]], dim=2)
            key = torch.cat([apply_rotary_emb(key[:, :, :-t], image_rotary_emb), key[:, :, -t:]], dim=2)
        else:
            query = apply_rotary_emb(query, image_rotary_emb)
            key = apply_rotary_emb(key, image_rotary_emb)
        return query, key

    def _step_encoder_to_qkv_and_concat(self, attn, query, key, value, encoder_hidden_states):
        if attn.add_q_proj is not None:
            eq = attn.add_q_proj(encoder_hidden_states).unflatten(2, (attn.heads, -1)).transpose(1, 2)
            ek = attn.add_k_proj(encoder_hidden_states).unflatten(2, (attn.heads, -1)).transpose(1, 2)
            ev = attn.add_v_proj(encoder_hidden_states).unflatten(2, (attn.heads, -1)).transpose(1, 2)
            if attn.norm_added_q is not None:
                eq = attn.norm_added_q(eq)
            if attn.norm_added_k is not None:
                ek = attn.norm_added_k(ek)
            query = torch.cat([query, eq], dim=2)
            key = torch.cat([key, ek], dim=2)
            value = torch.cat([value, ev], dim=2)
        return query, key, value

    # ---- step 5: attention --------------------------------------------------------------------------
    def _joint_attention(self, query, key, value, plan: ops.Plan, text_len: int, branch=None, weights=None,
                         flags: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
        """[video | text] joint attention for every branch in one C-ABI call; returns (video, text) outputs.
        Under Ulysses the video part is exchanged (once for all branches), each rank keeps its head slice of the
        replicated text tokens and the text outputs are all-gathered over heads (hunyuan.py:147-164,184-187)."""
        B = query.shape[0]
        assert B == 1, f"Batch size {B} is not supported for {self.__class__.__name__}."        # hunyuan.py:168
        return routed_attention(plan, query, key, value, branch=branch, weights=weights, flags=flags, text_len=text_len)

    def _step_attention(self, query, key, value, attention_mask, encoder_hidden_states_seq_len: int,
                        skip_communication: bool = False, text_valid: Optional[int] = None
                        ) -> Tuple[torch.Tensor, torch.Tensor]:
        """Full attention over the first S + valid_text tokens, zeros for padded text rows (hunyuan.py:136-189)."""
        text_len = encoder_hidden_states_seq_len
        video_len = (query.shape[2] - text_len) * (SP_STATE.sp_size if SP_STATE.enabled and not skip_communication else 1)
        if text_valid is None:
            text_valid = _valid_text(attention_mask, video_len)
        plan = get_plan((1, 1, video_len), (1, 1, video_len), (1, 1, 1), (1, 1, 1), 0, text_len, text_valid)
        H = query.shape[1]
        return self._joint_attention(query, key, value, plan, text_len, branch=[L.BRANCH_FULL] * H)

    def _step_to_output(self, attn, hidden_states, encoder_hidden_states):
        hidden_states = hidden_states.transpose(1, 2).flatten(2, 3)
        encoder_hidden_states = encoder_hidden_states.transpose(1, 2).flatten(2, 3)
        if getattr(attn, "to_out", None) is not None:
            hidden_states = attn.to_out[0](hidden_states)
            hidden_states = attn.to_out[1](hidden_states)
        if getattr(attn, "to_add_out", None) is not None:
            encoder_hidden_states = attn.to_add_out(encoder_hidden_states)
        return hidden_states, encoder_hidden_states

    def _qkv_fused(self, attn, hidden_states, encoder_hidden_states, image_rotary_emb):
        """Steps 1-4 (hunyuan.py:42-134) with ONE elementwise pass per Q / K stream: the projection GEMMs write
        (B, rows, H*128); ``vb_block_headnorm_rope`` applies the per-head RMSNorm, rotates the video rows and places
        the rows in the joint [video | text] tensor; V is written into it by the GEMM itself.  None = not applicable
        (other norm modules, dtypes, devices): the eager steps run instead."""
        norms = [_head_norm(getattr(attn, n, None)) for n in ("norm_q", "norm_k", "norm_added_q", "norm_added_k")]
        wants_grad = torch.is_grad_enabled() and (hidden_states.requires_grad or encoder_hidden_states.requires_grad
                                                  or attn.to_q.weight.requires_grad)
        if (hidden_states.dtype != torch.bfloat16 or not hidden_states.is_cuda or hidden_states.dim() != 3
                or any(n is False for n in norms) or wants_grad):      # the fused kernels are forward-only
            return None
        (wq, eq_), (wk, ek_), (waq, eaq), (wak, eak) = norms
        B, S, _ = hidden_states.shape
        T = encoder_hidden_states.shape[1]
        H = attn.heads
        cos, sin = _rope_tables(image_rotary_emb)
        hidden_states = hidden_states.contiguous()
        encoder_hidden_states = encoder_hidden_states.contiguous()
        if attn.add_q_proj is None:
            # single-stream block: one projection over the joint sequence, norm everywhere, RoPE on the video rows
            joint = torch.cat([hidden_states, encoder_hidden_states], dim=1)
            query = ops.headnorm_rope(attn.to_q(joint), wq, eq_, H, cos, sin, rope_rows=S)
            key = ops.headnorm_rope(attn.to_k(joint), wk, ek_, H, cos, sin, rope_rows=S)
            value = attn.to_v(joint)
        else:
            dim = H * 128
            query = torch.empty((B, S + T, dim), dtype=hidden_states.dtype, device=hidden_states.device)
            key, value = torch.empty_like(query), torch.empty_like(query)
            ops.headnorm_rope(attn.to_q(hidden_states), wq, eq_, H, cos, sin, out=query)
            ops.headnorm_rope(attn.to_k(hidden_states), wk, ek_, H, cos, sin, out=key)
            ops.headnorm_rope(attn.add_q_proj(encoder_hidden_states), waq, eaq, H, out=query, dst_row0=S)
            ops.headnorm_rope(attn.add_k_proj(encoder_hidden_states), wak, eak, H, out=key, dst_row0=S)
            for b in range(B):
                _linear_into(attn.to_v, hidden_states[b], value[b, :S])
                _linear_into(attn.add_v_proj, encoder_hidden_states[b], value[b, S:])
        return tuple(t.unflatten(2, (H, -1)).transpose(1, 2) for t in (query, key, value))

    def _qkv(self, attn, hidden_states, encoder_hidden_states, image_rotary_emb):
        fused = self._qkv_fused(attn, hidden_states, encoder_hidden_states, image_rotary_emb)
        if fused is not None:
            return fused
        query, key, value = self._step_to_qkv_and_unflatten(attn, hidden_states, encoder_hidden_states)
        query, key = self._step_qk_norm(attn, query, key)
        query, key = self._step_rotary_emb(attn, query, key, encoder_hidden_states.shape[1], image_rotary_emb)
        return self._step_encoder_to_qkv_and_concat(attn, query, key, value, encoder_hidden_states)

    def __call__(self, attn, hidden_states, encoder_hidden_states, attention_mask, image_rotary_emb,
                 text_valid: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """``text_valid`` (extra, optional): the number of un-padded text tokens when the caller already knows it —
        the reference reads it from ``attention_mask`` with a host sync in every layer (hunyuan.py:169)."""
        query, key, value = self._qkv(attn, hidden_states, encoder_hidden_states, image_rotary_emb)
        hidden_states, encoder_hidden_states = self._step_attention(
            query, key, value, attention_mask, encoder_hidden_states.shape[1], text_valid=text_valid)
        return self._step_to_output(attn, hidden_states, encoder_hidden_states)


class HunyuanVideoFlashAttnProcessorTripleTrain(HunyuanVideoFlashAttnProcessor):
    def __init__(self, check_input: bool = False):
        super().__init__()
        self.check_input = check_input

    def _check_input(self, hidden_states, lowres_group_info, latent_shape, window_size, tile_size):
        """Same checks, same messages as hunyuan.py:247-272."""
        if self.check_input:
            seq_length = hidden_states.shape[1] * SP_STATE.sp_size
            num_groups = lowres_group_info.center_indices.shape[0]
            group_size = lowres_group_info.center_indices.shape[1] + lowres_group_info.margin_indices.shape[1]
            if seq_length != latent_shape[0] * latent_shape[1] * latent_shape[2]:
                raise ValueError(f"Input sequence length {seq_length} does not match latent shape {latent_shape}.")
            for t_size, l_size in zip(tile_size, latent_shape):
                if l_size % t_size != 0:
                    raise ValueError(f"Tile size {tile_size} (dim={t_size}) does not divide latent shape "
                                     f"{latent_shape} (dim={l_size}).")
            if seq_length != num_groups * group_size:
                raise ValueError(f"Input sequence length {seq_length} does not match low-res info "
                                 f"{num_groups}x{group_size}.")

    def _plan(self, lowres_group_info, window_size, tile_size, latent_shape, text_len, attention_mask,
              text_valid: Optional[int] = None) -> ops.Plan:
        S = latent_shape[0] * latent_shape[1] * latent_shape[2]
        lowres_window = infer_lowres_window(lowres_group_info, latent_shape)
        if text_valid is None:
            text_valid = _valid_text(attention_mask, S)
        return get_plan(latent_shape, tile_size, window_size, lowres_window,
                        lowres_group_info.num_unpooled_tokens_per_group, text_len, text_valid)

    def _routed(self, attn, hidden_states, encoder_hidden_states, attention_mask, image_rotary_emb, lowres_group_info,
                window_size, tile_size, latent_shape, branch=None, weights=None, text_valid=None):
        self._check_input(hidden_states, lowres_group_info, latent_shape, window_size, tile_size)
        text_len = encoder_hidden_states.shape[1]
        query, key, value = self._qkv(attn, hidden_states, encoder_hidden_states, image_rotary_emb)
        plan = self._plan(lowres_group_info, window_size, tile_size, latent_shape, text_len, attention_mask, text_valid)
        # K and V are pooled with K's own matching, the output is unpooled with Q's (hunyuan.py:433-451)
        video, text = self._joint_attention(query, key, value, plan, text_len, branch=branch, weights=weights,
                                            flags=L.ATTN_CORESET_KV_FROM_K)
        return self._step_to_output(attn, video, text)

    def __call__(self, attn, hidden_states, encoder_hidden_states, attention_mask, image_rotary_emb,
                 use_original_attn: bool = False, routing_score: Optional[torch.Tensor] = None,
                 lowres_group_info: Optional[LowresGroupInfo] = None, flex_attn_mask_func: Optional[Callable] = None,
                 window_size: Tuple[int, int, int] = (3, 3, 3), tile_size: Tuple[int, int, int] = (6, 8, 8),
                 latent_shape: Tuple[int, int, int] = (30, 48, 80), text_valid: Optional[int] = None
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
        if use_original_attn:
            return HunyuanVideoFlashAttnProcessor.__call__(self, attn, hidden_states, encoder_hidden_states,
                                                           attention_mask, image_rotary_emb, text_valid=text_valid)
        return self._routed(attn, hidden_states, encoder_hidden_states, attention_mask, image_rotary_emb,
                            lowres_group_info, window_size, tile_size, latent_shape, weights=routing_score,
                            text_valid=text_valid)


class HunyuanVideoFlashAttnProcessorTripleEval(HunyuanVideoFlashAttnProcessorTripleTrain):
    @torch.no_grad()
    def __call__(self, attn, hidden_states, encoder_hidden_states, attention_mask, image_rotary_emb,
                 routing_score: torch.Tensor, tau_sparse: float, lowres_group_info: Optional[LowresGroupInfo] = None,
                 flex_attn_mask_func: Optional[Callable] = None, window_size: Tuple[int, int, int] = (3, 3, 3),
                 tile_size: Tuple[int, int, int] = (6, 8, 8), latent_shape: Tuple[int, int, int] = (30, 48, 80),
                 branch: Optional[Sequence[int]] = None, text_valid: Optional[int] = None
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
        if branch is None:
            branch = _top1_branches(routing_score, tau_sparse)          # hunyuan.py:620-624
        return self._routed(attn, hidden_states, encoder_hidden_states, attention_mask, image_rotary_emb,
                            lowres_group_info, window_size, tile_size, latent_shape, branch=branch,
                            text_valid=text_valid)
