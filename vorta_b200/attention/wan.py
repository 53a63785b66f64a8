"""Wan 2.1 attention processors — the reference's ``vorta/attention/wan.py`` interface on the sm_100a kernels.

Class names, ``__call__`` signatures, defaults and error behaviour follow the reference
(WanAttnProcessor2_0 :40-160, WanAttnProcessorTripleTrain :163-300, WanAttnProcessorTripleEval :303-438) so
``apply_vorta_transformer`` can install them unchanged.  What differs is underneath:

* the three branches, the head split (``_get_routed_qkv`` :388-416), the recombination (:418-438) and the Train
  blend (:296-300) are ONE call into ``vb_attn_fwd`` — heads carry their branch id, nothing is gathered by head;
* Q, K, V stay in the (B, S, H, D) memory the projections produce; the kernels read it through strides;
* under Ulysses, Q/K/V cross the NVLink fabric once for all branches (the reference sends them once per branch).

The projections / RMSNorm / RoPE in ``_input_proj`` are library calls (cuBLAS GEMMs and elementwise torch ops) as
in the reference; fusing them is the first "next" row of SURVEY.md section 8f.
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence, Tuple

import torch

from .. import _lib as L
from .. import ops
from ..ulysses import SP_STATE, exchange_out, exchange_qkv, shrink_dim
from ..ulysses.routed import routed_attention
from ._plans import get_plan, infer_lowres_window
from .coreset_select import LowresGroupInfo


def apply_rotary_emb(hidden_states: torch.Tensor, freqs: torch.Tensor) -> torch.Tensor:
    """Complex rotation of channel pairs (wan.py:34-37).  The reference multiplies in complex128; fp32 is used
    here — RoPE sits outside the bit-exact contract (SURVEY.md section 7.3 item 8)."""
    x = torch.view_as_complex(hidden_states.float().unflatten(3, (-1, 2)))
    out = torch.view_as_real(x * freqs.to(torch.complex64)).flatten(3, 4)
    return out.type_as(hidden_states)


_ROPE_CACHE = {}


def _rope_tables(rotary_emb: torch.Tensor):
    """fp32 (S_loc, 64) cos / sin tables of a complex (1, 1, S_loc, 64) phase tensor; the same tensor object is
    handed to every block of a forward, so the last conversion is cached."""
    key = (rotary_emb.data_ptr(), tuple(rotary_emb.shape), rotary_emb.storage_offset())
    hit = _ROPE_CACHE.get("last")
    if hit is not None and hit[0] == key:
        return hit[1], hit[2]
    r = rotary_emb.reshape(rotary_emb.shape[-2], rotary_emb.shape[-1])
    cos, sin = r.real.float().contiguous(), r.imag.float().contiguous()
    _ROPE_CACHE["last"] = (key, cos, sin, rotary_emb)       # keep the source alive so the pointer stays unique
    return cos, sin


def _norm_rope(norm, x: torch.Tensor, cos, sin) -> torch.Tensor:
    """norm_q / norm_k (RMSNorm across heads) followed by RoPE, fused; plain RoPE when the module has no norm."""
    if norm is not None and getattr(norm, "weight", None) is not None and x.is_contiguous():
        eps = norm.eps if getattr(norm, "eps", None) is not None else torch.finfo(x.dtype).eps
        return ops.rmsnorm_rope(x, norm.weight, eps, cos, sin)
    if norm is not None:
        x = norm(x)
    if cos is not None:
        heads = x.shape[-1] // 128
        x = apply_rotary_emb(x.unflatten(2, (heads, -1)).transpose(1, 2),
                             torch.complex(cos, sin)[None, None]).transpose(1, 2).flatten(2, 3)
    return x


def _top1_branches(routing_score: torch.Tensor, tau_sparse: Optional[float]) -> Sequence[int]:
    """wan.py:396-400: the first sample's top-1 expert per head; below ``tau_sparse`` -> full attention."""
    score, idx = routing_score[0].float().topk(1, dim=-1)
    idx = idx.clone()
    if tau_sparse is not None:
        idx[score < tau_sparse] = 0
    return idx.squeeze(-1).tolist()


class WanAttnProcessor2_0:
    def __init__(self):
        L.lib()      # fail loudly at construction if the CUDA library is missing: there is no fallback

    def __call__(self, attn, hidden_states: torch.Tensor, encoder_hidden_states: Optional[torch.Tensor] = None,
                 attention_mask: Optional[torch.Tensor] = None, rotary_emb: Optional[torch.Tensor] = None
                 ) -> torch.Tensor:
        is_cross_attn = encoder_hidden_states is not None
        query, key, value, encoder_hidden_states_img = self._input_proj(
            attn, hidden_states, encoder_hidden_states, rotary_emb)
        hidden_states, hidden_states_img = self._attn(
            attn, query, key, value, attention_mask, encoder_hidden_states_img, is_cross_attn)
        return self._output_proj(attn, hidden_states, hidden_states_img)

    def _input_proj(self, attn, hidden_states, encoder_hidden_states=None, rotary_emb=None):
        encoder_hidden_states_img = None
        if getattr(attn, "add_k_proj", None) is not None:
            encoder_hidden_states_img = encoder_hidden_states[:, :257]      # wan.py:74-76 (I2V image tokens)
            encoder_hidden_states = encoder_hidden_states[:, 257:]
        if encoder_hidden_states is None:
            encoder_hidden_states = hidden_states
        query = attn.to_q(hidden_states)
        key = attn.to_k(encoder_hidden_states)
        value = attn.to_v(encoder_hidden_states)
        cos = sin = None
        if rotary_emb is not None:
            cos, sin = _rope_tables(shrink_dim(rotary_emb, dim=2))
        # RMSNorm across heads + RoPE in one pass per tensor (reference: bf16 RMSNorm, then complex128 RoPE)
        query = _norm_rope(attn.norm_q, query, cos, sin)
        key = _norm_rope(attn.norm_k, key, cos, sin)
        # (B, S, H*D) -> (B, H, S, D) as a VIEW: the kernels take the strides
        query = query.unflatten(2, (attn.heads, -1)).transpose(1, 2)
        key = key.unflatten(2, (attn.heads, -1)).transpose(1, 2)
        value = value.unflatten(2, (attn.heads, -1)).transpose(1, 2)
        return query, key, value, encoder_hidden_states_img

    def _attn(self, attn, query, key, value, attention_mask, encoder_hidden_states_img, is_cross_attn: bool,
              skip_communication: bool = False) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        if attention_mask is not None:
            raise ValueError("attention_mask is not supported by the Wan processors (the reference passes None)")
        sp = SP_STATE.enabled and not skip_communication
        if sp and not is_cross_attn:
            query, key, value = exchange_qkv(query, key, value)
        # cross attention under SP: every rank keeps its own queries and all heads of the replicated text K/V —
        # the same function as the reference's Q all-to-all + K/V head slice (wan.py:110-114) with no traffic
        hidden_states_img = None
        if encoder_hidden_states_img is not None:
            key_img = attn.norm_added_k(attn.add_k_proj(encoder_hidden_states_img))
            value_img = attn.add_v_proj(encoder_hidden_states_img)
            key_img = key_img.unflatten(2, (attn.heads, -1)).transpose(1, 2)
            value_img = value_img.unflatten(2, (attn.heads, -1)).transpose(1, 2)
            hidden_states_img = ops.attn_dense(query, key_img, value_img)
        hidden_states = ops.attn_dense(query, key, value)
        if sp and not is_cross_attn:
            hidden_states = exchange_out(hidden_states)
        return hidden_states, hidden_states_img

    def _output_proj(self, attn, hidden_states, hidden_states_img):
        hidden_states = hidden_states.transpose(1, 2).flatten(2, 3)           # free: memory is (B, S, H, D)
        if hidden_states_img is not None:
            hidden_states = hidden_states + hidden_states_img.transpose(1, 2).flatten(2, 3)
        hidden_states = attn.to_out[0](hidden_states)
        hidden_states = attn.to_out[1](hidden_states)
        return hidden_states


class WanAttnProcessorTripleTrain(WanAttnProcessor2_0):
    def __init__(self, check_input: bool = False):
        super().__init__()
        self.check_input = check_input

    def _check_input(self, hidden_states, lowres_group_info, latent_shape, window_size, tile_size):
        """Same checks, same messages as wan.py:168-193."""
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

    @staticmethod
    def _plan(lowres_group_info, flex_attn_mask_func, window_size, tile_size, latent_shape) -> ops.Plan:
        # ``flex_attn_mask_func`` (a BlockMask in the reference) is accepted and not needed: the schedule is
        # derived from (latent_shape, window_size, tile_size) — SURVEY.md section 8b "kwargs objects"
        lowres_window = infer_lowres_window(lowres_group_info, latent_shape)
        return get_plan(latent_shape, tile_size, window_size, lowres_window,
                        lowres_group_info.num_unpooled_tokens_per_group)

    def _routed_attention(self, query, key, value, plan: ops.Plan, branch=None, weights=None) -> torch.Tensor:
        """All branches of one layer: a single C-ABI call between the two Ulysses exchanges."""
        return routed_attention(plan, query, key, value, branch=branch, weights=weights)[0]

    def __call__(self, attn, hidden_states: torch.Tensor, encoder_hidden_states: Optional[torch.Tensor] = None,
                 attention_mask: Optional[torch.Tensor] = None, rotary_emb: Optional[torch.Tensor] = None,
                 use_original_attn: bool = False, routing_score: Optional[torch.Tensor] = None,
                 lowres_group_info: Optional[LowresGroupInfo] = None,
                 flex_attn_mask_func: Optional[Callable] = None,
                 window_size: Tuple[int, int, int] = (3, 3, 3), tile_size: Tuple[int, int, int] = (6, 8, 8),
                 latent_shape: Tuple[int, int, int] = (20, 30, 52)) -> torch.Tensor:
        is_cross_attn = encoder_hidden_states is not None
        if is_cross_attn or use_original_attn:
            return WanAttnProcessor2_0.__call__(self, attn, hidden_states, encoder_hidden_states, attention_mask,
                                                rotary_emb)
        self._check_input(hidden_states, lowres_group_info, latent_shape, window_size, tile_size)
        query, key, value, _ = self._input_proj(attn, hidden_states, encoder_hidden_states=None, rotary_emb=rotary_emb)
        plan = self._plan(lowres_group_info, flex_attn_mask_func, window_size, tile_size, latent_shape)
        # every branch on every head, out = sum_e score[b, h, e] * O_e (wan.py:227-239, :296-300), fused in the
        # attention epilogue
        hidden_states = self._routed_attention(query, key, value, plan, weights=routing_score)
        return self._output_proj(attn, hidden_states, hidden_states_img=None)


class WanAttnProcessorTripleEval(WanAttnProcessorTripleTrain):
    @torch.no_grad()
    def __call__(self, attn, hidden_states: torch.Tensor, encoder_hidden_states: torch.Tensor,
                 attention_mask: torch.Tensor, rotary_emb: torch.Tensor, tau_sparse: float,
                 routing_score: torch.Tensor, lowres_group_info: Optional[LowresGroupInfo] = None,
                 flex_attn_mask_func: Optional[Callable] = None,
                 window_size: Tuple[int, int, int] = (3, 3, 3), tile_size: Tuple[int, int, int] = (6, 8, 8),
                 latent_shape: Tuple[int, int, int] = (20, 30, 52), use_original_attn: bool = False,
                 branch: Optional[Sequence[int]] = None):
        """``branch`` (extra, optional): per-head branch ids already decided for this layer — the router of every
        layer only depends on the timestep embedding, so a caller can decide a whole step's routing in one
        ``router_forward`` launch + one device->host copy instead of one sync per layer (wan.py:409)."""
        is_cross_attn = encoder_hidden_states is not None
        if is_cross_attn or use_original_attn:
            return WanAttnProcessor2_0.__call__(self, attn, hidden_states, encoder_hidden_states, attention_mask,
                                                rotary_emb)
        self._check_input(hidden_states, lowres_group_info, latent_shape, window_size, tile_size)
        if branch is None:
            branch = _top1_branches(routing_score, tau_sparse)
        plan = self._plan(lowres_group_info, flex_attn_mask_func, window_size, tile_size, latent_shape)
        query, key, value, _ = self._input_proj(attn, hidden_states, encoder_hidden_states=None, rotary_emb=rotary_emb)
        hidden_states = self._routed_attention(query, key, value, plan, branch=branch)
        return self._output_proj(attn, hidden_states, hidden_states_img=None)
