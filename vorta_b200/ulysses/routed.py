"""One routed attention layer under sequence parallelism, for both the Wan and the HunyuanVideo processors.

Without SP this is one ``vb_attn_fwd`` call.  With SP, the top-1 (Eval) routing at batch size 1 takes the NVLink
peer-memory exchange (``peer.py``) with the unit placement of ``balance.layer_placement``; blend (Train) mode, larger
batches, ``VB_ULYSSES=nccl`` and boxes without peer memory take the NCCL all-to-all (``utils.py``) with the head table
of ``balance.balance_heads``.  HunyuanVideo's replicated text rows (``text_len`` of them, behind the video rows) are
not exchanged: every rank attends with its heads' text rows, and the text outputs are gathered over heads.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from .. import _lib as L
from .. import ops
from . import balance, peer
from .parallel_states import SP_STATE
from .utils import all_gather, exchange_out, exchange_qkv, local_heads, shrink_dim


def local_units(placement, rank: int, branch: Sequence[int], slots: int):
    """(branch id per slot, output head per slot) of this rank for ``vb_attn_fwd``: unused slots are skipped, the parts
    of a split full head become VB_BRANCH_FULL_PART(k, n)."""
    ids, out_heads = [], []
    for h, part in placement[rank]:
        e = int(branch[h])
        if part != balance.WHOLE:
            if e != L.BRANCH_FULL:
                raise ValueError("only full-attention heads are split into query parts")
            e = L.branch_full_part(*balance.part_kn(part))
        ids.append(e)
        out_heads.append(int(h))
    pad = slots - len(ids)
    return ids + [L.BRANCH_SKIP] * pad, out_heads + [0] * pad


def _split(out: torch.Tensor, text_len: int):
    n = out.shape[2] - text_len
    return out[:, :, :n], (out[:, :, n:] if text_len else None)


def routed_attention(plan: ops.Plan, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *,
                     branch: Optional[Sequence[int]] = None, weights: Optional[torch.Tensor] = None, flags: int = 0,
                     text_len: int = 0) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """-> (video, text). video: (B, H, S_loc, 128) view of (B, S_loc, H, 128) memory (S_loc = S without SP);
    text: (B, H, text_len, 128), or None when text_len == 0.

    q, k, v: (B, H, S_loc + text_len, 128) views: this rank's video tokens, then the replicated text tokens.
    ``branch`` / ``weights``: per-head branch ids (top-1) or (B, H, 3) routing scores (blend), as in
    ``ops.routed_attention``."""
    if not SP_STATE.enabled:
        return _split(ops.routed_attention(plan, q, k, v, branch=branch, weights=weights, flags=flags), text_len)
    B, H, N = q.shape[:3]
    n = N - text_len
    P, r = SP_STATE.sp_size, SP_STATE.group_local_rank
    ex = peer.get_exchange(H, n, q.device, text_len) if weights is None and B == 1 else None
    if ex is not None:
        # Q / K / V rows are stored straight into the buffers of the ranks that own the head (or a query half of it),
        # the attention epilogue stores every output row straight into the buffer of the rank that owns the token (text
        # rows to every rank); all ranks derive the same placement from the layer's routing
        placement = balance.layer_placement(branch, plan, P, ex.slots)
        if text_len:
            q, k, v = ex.scatter_qkv(q[:, :, :n], k[:, :, :n], v[:, :, :n], placement,
                                     text=[t[:, :, n:] for t in (q, k, v)])
            ex.zero_padded_text(plan.text_valid)
        else:
            q, k, v = ex.scatter_qkv(q, k, v, placement)
        ids, out_heads = local_units(placement, r, branch, ex.slots)
        ops.routed_attention(plan, q, k, v, branch=ids, flags=flags, out_peers=ex.out_ptrs, out_peer_rows=ex.s_loc,
                             out_peer_strides=(0, 128, H * 128), out_heads=out_heads)
        return _split(ex.finish_out(), text_len)

    head_at = None
    if branch is not None:
        # only slot numbers inside the exchange change: rank r holds heads head_at[r * H/P:(r + 1) * H/P]
        head_at = balance.balance_heads(list(branch), balance.branch_costs(plan), P)
        branch = local_heads(list(branch), H, head_at)
    if weights is not None:
        weights = shrink_dim(weights, dim=1)
    qs, ks, vs = exchange_qkv(q[:, :, :n], k[:, :, :n], v[:, :, :n], extra_rows=text_len, head_at=head_at)
    if text_len:
        mine = None if head_at is None else torch.tensor(local_heads(head_at, H), device=q.device)
        for dst, src in ((qs, q), (ks, k), (vs, v)):
            text = src[:, :, n:]
            dst[:, :, -text_len:] = shrink_dim(text, dim=1) if mine is None else text.index_select(1, mine)
    video, text = _split(ops.routed_attention(plan, qs, ks, vs, branch=branch, weights=weights, flags=flags), text_len)
    video = exchange_out(video, head_at)
    if text_len:
        text = all_gather(text.contiguous(), dim=1)
        if head_at is not None:       # gathered in slot order: put every head back at its own index
            inverse = torch.empty(H, dtype=torch.long)
            inverse[torch.tensor(head_at)] = torch.arange(H)
            text = text.index_select(1, inverse.to(text.device))
    return video, text
