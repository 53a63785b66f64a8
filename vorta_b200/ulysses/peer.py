"""Ulysses exchange over NVLink / NVSwitch peer memory, fused into the kernels on either side of the attention.

The reference (vorta/ulysses/utils.py:15-93) and the NCCL path of this package move Q, K, V and O with all-to-all
collectives plus layout copies.  Here every rank maps every peer's receive buffers (torch symmetric memory, one
allocation per geometry) and

  * "in"  : ``vb_ulysses_scatter_qkv_slots`` stores each (token, head) row of Q, K, V straight into the buffer of the
            rank that owns the head — one pass, no staging buffer, no collective;
  * "out" : the attention kernel's epilogue stores each output row straight into the buffer of the rank that owns the
            token (``vb_attn_args.out_peer_ptrs``), already in the (S_loc, H, 128) layout the output projection reads.

Two device-side barriers per layer order the remote stores against their consumers (see ``PeerExchange``).  Used for
the top-1 (Eval) processors at batch size 1, Wan and HunyuanVideo (whose replicated text rows are filled locally on the
way in and stored to every rank on the way out); the blended (Train) processors and larger batches take the NCCL path
in ``utils.py``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from .. import _lib as L
from . import balance
from .parallel_states import SP_STATE

_EXCHANGES: Dict[tuple, "PeerExchange"] = {}
_DISABLED_REASON: Optional[str] = None


class PeerExchange:
    """Symmetric receive buffers of one geometry (heads H, local tokens S_loc, world P), all 128-channel bf16:
    ``qkv`` (3, S + T, H/P, 128): this rank's head chunk over the full sequence, video rows written by every peer,
                                  the T replicated text rows (HunyuanVideo; T = 0 for Wan) filled locally;
    ``out`` (S_loc + T, H, 128): this rank's token shard over all heads, written by every peer's attention epilogue;
                                  text rows of every head are stored to every rank (the head all-gather of
                                  vorta/attention/hunyuan.py:186-187).

    Ordering per layer (all on the caller's stream):
        scatter_qkv -> barrier A -> attention (reads qkv, stores into peers' out) -> barrier B -> consumer reads out.
    A rank leaves barrier B only after every rank finished its attention, so the next layer's scatter cannot overwrite
    a qkv buffer that is still being read; it reaches the next barrier A only after its own consumer of ``out`` was
    issued, so nobody stores into ``out`` while it is still needed."""

    def __init__(self, heads: int, s_loc: int, device: torch.device, text_len: int = 0):
        import torch.distributed._symmetric_memory as symm
        P, rank = SP_STATE.sp_size, SP_STATE.group_local_rank
        self.P, self.rank, self.heads, self.s_loc, self.hp = P, rank, heads, s_loc, heads // P
        self.S = s_loc * P
        self.text_len = int(text_len)
        # head slots of the receive buffer: more than H / P, so that a rank can hold an uneven number of heads and
        # query halves of full heads (balance.place_units)
        self.slots = balance.max_slots(heads, P)
        group = SP_STATE.group if SP_STATE.group is not None else dist.group.WORLD
        self.qkv = symm.empty((3, self.S + self.text_len, self.slots, 128), dtype=torch.bfloat16, device=device)
        self.out = symm.empty((s_loc + self.text_len, heads, 128), dtype=torch.bfloat16, device=device)
        self.h_qkv = symm.rendezvous(self.qkv, group)
        self.h_out = symm.rendezvous(self.out, group)
        self.qkv_ptrs = (C.c_void_p * P)(*[int(p) for p in self.h_qkv.buffer_ptrs])
        self.out_ptrs = [int(p) for p in self.h_out.buffer_ptrs]
        # bytes this rank stores into OTHER ranks' buffers over NVLink, counted from the placement tables (the NVLink data
        # counters of nvidia-smi read N/A on this pool): "in" = Q/K/V rows of scatter_qkv, "out" = attention output rows
        self.nvlink_tx_bytes = 0

    def _tables(self, placement):
        peers, slots, heads = [], [], []
        for p, units in enumerate(placement):
            if len(units) > self.slots:
                raise ValueError(f"rank {p} was given {len(units)} units for {self.slots} slots")
            for slot, (h, _part) in enumerate(units):
                peers.append(p); slots.append(slot); heads.append(int(h))
        n = len(peers)
        remote_in = sum(1 for p in peers if p != self.rank)
        frac_out = sum(1.0 if part == balance.WHOLE else 1.0 / balance.part_kn(part)[1] for _, part in placement[self.rank])
        self.nvlink_tx_bytes += 3 * self.s_loc * remote_in * 256 + int(frac_out * (self.S - self.s_loc) * 256)
        arr = C.c_int32 * n
        return arr(*peers), arr(*slots), arr(*heads), n

    def _scatter(self, tensors, tables) -> None:
        """tensors: [q, k, v] (1, H, S_loc, 128) views."""
        i64x3 = C.c_int64 * 3
        ref = tensors[0]
        st_s = i64x3(*[t.stride(2) for t in tensors])
        st_h = i64x3(*[t.stride(1) for t in tensors])
        peers, slots, heads, n = tables
        with torch.cuda.device(ref.device):
            L.check(L.lib().vb_ulysses_scatter_qkv_slots(
                *[t.data_ptr() for t in tensors], st_s, st_h, self.qkv_ptrs, self.S + self.text_len, self.s_loc,
                self.slots, self.P, self.rank, peers, slots, heads, n, torch.cuda.current_stream(ref.device).cuda_stream))

    def scatter_qkv(self, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
                    placement: Sequence[Sequence[Tuple[int, int]]], text: Optional[Sequence[torch.Tensor]] = None
                    ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """q, k, v: (1, H, S_loc, 128) views of this rank's token shard.  ``placement[p]`` = the (head, part) units of
        rank p in slot order (``balance.layer_placement``); every head of a unit is stored into that slot of rank p's
        buffer — a head split into query parts goes to several ranks.  Returns (1, slots, S + T, 128) views of the
        local receive buffer, valid after barrier A (issued here); only the first len(placement[rank]) slots hold data.
        ``text``: the replicated (1, H, T, 128) text rows of q, k, v; the rows of this rank's heads are copied behind
        the video rows locally (no traffic)."""
        self._scatter([q, k, v], self._tables(placement))
        if self.text_len:
            mine = [h for h, _ in placement[self.rank]]
            sel = torch.tensor(mine, device=q.device)
            for i, t in enumerate(text):          # (1, H, T, 128) -> rows [S, S + T) of my first len(mine) slots
                self.qkv[i, self.S:, :len(mine)].copy_(t[0].index_select(0, sel).transpose(0, 1))
        self.h_qkv.barrier(channel=0)
        return tuple(self.qkv[i].unsqueeze(0).transpose(1, 2) for i in range(3))

    def zero_padded_text(self, text_valid: int) -> None:
        """Rows of padded text queries are written by nobody (hunyuan.py:176 pads with zeros): clear them locally."""
        if self.text_len > text_valid:
            self.out[self.s_loc + text_valid:].zero_()

    def finish_out(self) -> torch.Tensor:
        """Barrier B, then this rank's (1, H, S_loc + T, 128) view of the gathered outputs."""
        self.h_out.barrier(channel=1)
        return self.out.unsqueeze(0).transpose(1, 2)


def get_exchange(heads: int, s_loc: int, device: torch.device, text_len: int = 0) -> Optional[PeerExchange]:
    """The cached exchange for this geometry, or None when peer memory is unavailable / disabled
    (VB_ULYSSES=nccl), in which case the caller takes the NCCL path."""
    global _DISABLED_REASON
    if not SP_STATE.enabled or os.environ.get("VB_ULYSSES", "peer") == "nccl" or _DISABLED_REASON is not None:
        return None
    if SP_STATE.sp_size > 8 or heads % SP_STATE.sp_size != 0:
        return None
    key = (heads, s_loc, str(device), SP_STATE.sp_size, int(text_len))
    ex = _EXCHANGES.get(key)
    if ex is None:
        try:
            ex = PeerExchange(heads, s_loc, device, text_len)
        except Exception as e:                      # no P2P mapping on this box: say so once, use NCCL
            _DISABLED_REASON = f"{type(e).__name__}: {e}"
            if SP_STATE.rank == 0:
                print(f"vorta_b200.ulysses: peer-memory exchange unavailable ({_DISABLED_REASON}); using NCCL all-to-all",
                      flush=True)
            return None
        _EXCHANGES[key] = ex
    return ex


def disabled_reason() -> Optional[str]:
    return _DISABLED_REASON


def nvlink_tx_bytes(reset: bool = False) -> int:
    """Bytes this rank has stored into other ranks' exchange buffers since the last reset (all geometries)."""
    total = sum(ex.nvlink_tx_bytes for ex in _EXCHANGES.values())
    if reset:
        for ex in _EXCHANGES.values():
            ex.nvlink_tx_bytes = 0
    return total

