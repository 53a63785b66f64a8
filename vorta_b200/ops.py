"""Tensor-level wrappers over the C ABI: marshal torch tensors (pointers, strides, current stream) and nothing else.

No arithmetic on the path happens here; every function ends in a call into ``libvorta_b200.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib as L

HEAD_DIM = 128


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _require_cuda_bf16(name: str, t: torch.Tensor) -> None:
    if not t.is_cuda:
        raise L.VortaB200Error(f"{name} must be a CUDA tensor: vorta_b200 has no CPU path")
    if t.dtype != torch.bfloat16:
        raise ValueError(f"{name} must be bfloat16, got {t.dtype}")
    if t.dim() != 4 or t.shape[-1] != HEAD_DIM or t.stride(-1) != 1:
        raise ValueError(f"{name} must be (B, H, N, {HEAD_DIM}) with contiguous channels, got {tuple(t.shape)} "
                         f"strides {t.stride()}")


class Plan:
    """Geometry-only schedule shared by all layers: coreset groups, tile-major map, sliding-tile key runs.

    Mirrors what ``prepare_wan_self_attn_kwargs`` builds in the reference (vorta/patch/utils.py:8-36):
    ``get_group_info`` (coreset_select.py:15-60) and ``create_sliding_tile_attn_mask_func``
    (sliding_attn_flex.py:72-134) — here as closed-form tables, without a mask tensor.
    """

    def __init__(self, latent_shape: Sequence[int], tile_size: Sequence[int], window_size: Sequence[int],
                 lowres_window_size: Sequence[int], reduction_rate: float = 0.5, text_len: int = 0,
                 text_valid: int = 0, n_unpooled: Optional[int] = None):
        lib = L.lib()
        self.latent_shape = tuple(int(x) for x in latent_shape)
        self.tile_size = tuple(int(x) for x in tile_size)
        self.window_size = tuple(int(x) for x in window_size)
        self.lowres_window_size = tuple(int(x) for x in lowres_window_size)
        g = int(np.prod(self.lowres_window_size))
        if n_unpooled is None:
            # exactly the reference's expression (coreset_select.py:54), evaluated in Python floats
            n_unpooled = int(g * (1 - reduction_rate)) - 1
        desc = L.PlanDesc()
        desc.latent[:] = self.latent_shape
        desc.tile[:] = self.tile_size
        desc.window[:] = self.window_size
        desc.lowres_window[:] = self.lowres_window_size
        desc.n_unpooled = int(n_unpooled)
        desc.text_len = int(text_len)
        desc.text_valid = int(text_valid)
        handle = C.c_void_p()
        L.check(lib.vb_plan_create(C.byref(handle), C.byref(desc)))
        self._h = handle
        self.text_len = int(text_len)
        self.text_valid = int(text_valid)
        self.n_unpooled = int(n_unpooled)
        self.seq_len = self.query(L.PLAN_SEQ_LEN)
        self.num_groups = self.query(L.PLAN_NUM_GROUPS)
        self.group_size = self.query(L.PLAN_GROUP_SIZE)
        self.coreset_len = self.query(L.PLAN_CORESET_LEN)
        self.num_pooled = self.query(L.PLAN_NUM_POOLED)
        self.num_tiles = self.query(L.PLAN_NUM_TILES)
        self.tile_tokens = self.query(L.PLAN_TILE_TOKENS)
        self._ws = {}

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                L.lib().vb_plan_destroy(h)
            except Exception:
                pass
            self._h = None

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def query(self, what: int) -> int:
        v = C.c_int64()
        L.check(L.lib().vb_plan_query(self._h, what, C.byref(v)))
        return int(v.value)

    def export(self, what: int) -> np.ndarray:
        n = C.c_int64(0)
        L.check(L.lib().vb_plan_export(self._h, what, None, C.byref(n)))
        dtype = np.int64 if what in (L.EXPORT_CENTER_INDICES, L.EXPORT_MARGIN_INDICES) else np.int32
        buf = np.empty(n.value // np.dtype(dtype).itemsize, dtype=dtype)
        L.check(L.lib().vb_plan_export(self._h, what, buf.ctypes.data_as(C.c_void_p), C.byref(n)))
        return buf

    def set_text_valid(self, text_valid: int) -> None:
        L.check(L.lib().vb_plan_set_text_valid(self._h, int(text_valid)))
        self.text_valid = int(text_valid)

    def workspace(self, batch: int, heads: int, device: torch.device) -> torch.Tensor:
        need = int(L.lib().vb_attn_workspace_bytes(self._h, batch, heads))
        key = (str(device),)
        ws = self._ws.get(key)
        if ws is None or ws.numel() < need:
            ws = torch.empty(need, dtype=torch.uint8, device=device)
            self._ws[key] = ws
        return ws

    # flop formulas of BASELINE.md section 3 (per head), for reporting
    def flops_per_head(self, branch: int) -> float:
        S, tv, D = self.seq_len, self.text_valid, HEAD_DIM
        if branch == L.BRANCH_FULL:
            return 4.0 * (S + tv) ** 2 * D
        if branch == L.BRANCH_CORESET:
            return 4.0 * (self.coreset_len + tv) ** 2 * D
        kw = self.query(L.PLAN_KEYS_PER_QUERY)
        return 4.0 * D * (S * (kw + tv) + tv * (S + tv))


def routed_attention(plan: Plan, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
                     branch: Optional[Sequence[int]] = None, weights: Optional[torch.Tensor] = None,
                     flags: int = 0, out: Optional[torch.Tensor] = None,
                     debug: Optional[torch.Tensor] = None, out_peers: Optional[Sequence[int]] = None,
                     out_peer_rows: int = 0, out_peer_strides: Optional[Sequence[int]] = None,
                     head_offset: int = 0, out_heads: Optional[Sequence[int]] = None) -> Optional[torch.Tensor]:
    """One routed self-attention layer.  q, k, v: (B, H, S + text_len, 128) bf16 views (any batch / head / token
    strides).  ``branch``: per-head VB_BRANCH_* ids (Eval processor semantics, wan.py:388-438); ``weights``:
    (B, H, 3) routing scores for the blended Train semantics (wan.py:296-300).  Returns (B, H, N, 128) as a view
    of (B, N, H, 128) memory, so ``transpose(1, 2).flatten(2, 3)`` (wan.py:152) is free.
    ``out_heads``: head index along the output's head stride for each local head (default: ``head_offset + h``)."""
    for name, t in (("q", q), ("k", k), ("v", v)):
        _require_cuda_bf16(name, t)
    B, H, N, D = q.shape
    if N != plan.seq_len + plan.text_len:
        raise ValueError(f"Input sequence length {N} does not match latent shape {plan.latent_shape}"
                         f" (+ text {plan.text_len}).")
    if k.shape != q.shape or v.shape != q.shape:
        raise ValueError(f"q, k and v must have the same shape, got {tuple(q.shape)}, {tuple(k.shape)}, "
                         f"{tuple(v.shape)}")
    if out_heads is not None and (len(out_heads) != H or min(out_heads) < 0):
        raise ValueError(f"out_heads needs one non-negative output head per local head ({H}), got {list(out_heads)}")
    if out_peers is None and out is not None:
        _require_cuda_bf16("out", out)
        last = max(out_heads) if out_heads is not None else H - 1
        if out.shape[0] != B or out.shape[2] != N or out.shape[1] <= last:
            raise ValueError(f"out must be (B={B}, more than {last} heads, N={N}, {D}), got {tuple(out.shape)}")
    args = L.AttnArgs()
    if out_peers is not None:
        # fused Ulysses "out" exchange: rows go straight into the owner ranks' (S_loc, H_total, 128) buffers; local
        # head h lands at head out_heads[h] there
        out = None
        sb, sh, ss = out_peer_strides
        args.out = None
        args.out_stride[:] = (sb, sh, ss)
        for i, ptr in enumerate(out_peers):
            args.out_peer_ptrs[i] = int(ptr)
        if out_heads is None:
            out_heads = range(head_offset, head_offset + H)
        args.out_peer_count, args.out_peer_rows = len(out_peers), int(out_peer_rows)
    else:
        if out is None:
            out = torch.empty((B, N, H, D), dtype=q.dtype, device=q.device).transpose(1, 2)
        args.out = out.data_ptr()
        args.out_stride[:] = out.stride()[:3]
    args.q, args.k, args.v = q.data_ptr(), k.data_ptr(), v.data_ptr()
    args.q_stride[:] = q.stride()[:3]
    args.k_stride[:] = k.stride()[:3]
    args.v_stride[:] = v.stride()[:3]
    args.batch, args.heads = B, H
    keep = []
    if weights is not None:
        if weights.requires_grad and torch.is_grad_enabled():
            # the reference trains the routers through this blend (wan.py:296-300, scripts/wan/train_one_step.py);
            # the backward of the attention kernels is not built (DESIGN.md section 8), so refuse instead of
            # silently cutting the gradient
            raise NotImplementedError("vorta_b200: routed attention has no backward pass yet; run the Train "
                                      "processors under torch.no_grad() or detach the routing scores")
        if tuple(weights.shape) != (B, H, 3):
            raise ValueError(f"weights must be (B, H, 3), got {tuple(weights.shape)}")
        # the routing scores stay on the device (the reference blends device tensors, wan.py:296-300): no host sync
        w = weights.detach().to(device=q.device, dtype=torch.float32).contiguous()
        keep.append(w)
        args.weights = None
        args.weights_device = w.data_ptr()
    else:
        args.weights = None
        args.weights_device = None
    if branch is not None:
        br = (C.c_int32 * H)(*[int(x) for x in branch])
        keep.append(br)
        args.branch = C.cast(br, C.POINTER(C.c_int32))
    else:
        args.branch = None
    if out_heads is not None:
        oh = (C.c_int32 * H)(*[int(x) for x in out_heads])
        keep.append(oh)
        args.out_heads = C.cast(oh, C.POINTER(C.c_int32))
    else:
        args.out_heads = None
    args.flags = int(flags)
    ws = plan.workspace(B, H, q.device)
    args.workspace, args.workspace_bytes = ws.data_ptr(), ws.numel()
    args.debug = debug.data_ptr() if debug is not None else None
    with torch.cuda.device(q.device):
        L.check(L.lib().vb_attn_fwd(plan.handle, C.byref(args), _stream_ptr(q.device)))
    return out


def coreset_select(plan: Plan, x: torch.Tensor, want_tokens: bool = False):
    """Similarity selection of coreset_select.py:91-113 on (B, H, S[+text], 128) bf16.
    Returns (unpooled_argsort_sim, pooled_argsort_sim) int64 like ``MatchingResults`` and, when asked, the
    flat token tables the attention kernel consumes."""
    _require_cuda_bf16("x", x)
    B, H = x.shape[:2]
    G, n_u, n_p = plan.num_groups, plan.n_unpooled, plan.num_pooled
    dev = x.device
    un = torch.empty((B, H, G, n_u), dtype=torch.int64, device=dev)
    po = torch.empty((B, H, G, n_p), dtype=torch.int64, device=dev)
    kept = torch.empty((B, H, plan.coreset_len + plan.text_len), dtype=torch.int32, device=dev)
    drop = torch.empty((B, H, G, max(n_p, 1)), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.lib().vb_coreset_select(plan.handle, x.data_ptr(), x.stride(0), x.stride(1), x.stride(2), B, H,
                                          un.data_ptr(), po.data_ptr(), kept.data_ptr(), drop.data_ptr(),
                                          _stream_ptr(dev)))
    if want_tokens:
        return un, po, kept, drop[..., :n_p]
    return un, po


def gather_rows(src: torch.Tensor, row_map: torch.Tensor, n_rows: Optional[int] = None) -> torch.Tensor:
    """dst[b, h, i] = src[b, h, map[b, h, i]]; ``row_map`` int32 of shape (n,), (H, n) or (B, H, n)."""
    _require_cuda_bf16("src", src)
    B, H = src.shape[:2]
    if row_map.dtype != torch.int32 or not row_map.is_cuda:
        raise ValueError("row_map must be a CUDA int32 tensor")
    row_map = row_map.contiguous()
    n = int(row_map.shape[-1]) if n_rows is None else int(n_rows)
    if row_map.dim() == 1:
        sb, sh = 0, 0
    elif row_map.dim() == 2:
        sb, sh = 0, row_map.stride(0)
    else:
        sb, sh = row_map.stride(0), row_map.stride(1)
    dst = torch.empty((B, H, n, HEAD_DIM), dtype=src.dtype, device=src.device)
    with torch.cuda.device(src.device):
        L.check(L.lib().vb_gather_rows(src.data_ptr(), src.stride(0), src.stride(1), src.stride(2), dst.data_ptr(),
                                       dst.stride(0), dst.stride(1), dst.stride(2), row_map.data_ptr(), sb, sh,
                                       B, H, n, _stream_ptr(src.device)))
    return dst


def router_forward(temb: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, heads: int,
                   tau: Optional[float] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """softmax(W silu(temb) + b) in fp32 for L stacked routers (router.py:41-43) and the top-1 / threshold
    decision of wan.py:398-400.  temb (B, E); weight (L, 3H, E) or (3H, E); bias (L, 3H) or (3H,).
    Returns scores (L, B, H, 3) fp32 and branch ids (L, H) int32 (device tensors)."""
    if not temb.is_cuda:
        raise L.VortaB200Error("router_forward needs CUDA tensors: vorta_b200 has no CPU path")
    if weight.dim() == 2:
        weight, bias = weight.unsqueeze(0), bias.unsqueeze(0)
    if weight.dtype != bias.dtype:
        bias = bias.to(weight.dtype)
    codes = {torch.float32: L.DTYPE_F32, torch.bfloat16: L.DTYPE_BF16}
    if temb.dtype not in codes or weight.dtype not in codes:
        raise ValueError(f"router dtypes must be float32 or bfloat16, got {temb.dtype} / {weight.dtype}")
    temb, weight, bias = temb.contiguous(), weight.contiguous(), bias.contiguous()
    n_layers, n_out, E = weight.shape
    B = temb.shape[0]
    if n_out != 3 * heads or temb.shape[1] != E:
        raise ValueError(f"router shapes inconsistent: temb {tuple(temb.shape)}, weight {tuple(weight.shape)}")
    scores = torch.empty((n_layers, B, heads, 3), dtype=torch.float32, device=temb.device)
    branch = torch.empty((n_layers, heads), dtype=torch.int32, device=temb.device)
    with torch.cuda.device(temb.device):
        L.check(L.lib().vb_router_forward(temb.data_ptr(), codes[temb.dtype], weight.data_ptr(), bias.data_ptr(),
                                          codes[weight.dtype], weight.stride(0), bias.stride(0), n_layers, B, E,
                                          heads, float("nan") if tau is None else float(tau), scores.data_ptr(),
                                          branch.data_ptr(), _stream_ptr(temb.device)))
    return scores, branch


def stats_reset() -> None:
    L.lib().vb_stats_reset()


def stats() -> Tuple[int, float]:
    lib = L.lib()
    return int(lib.vb_stats_launches()), float(lib.vb_stats_attn_flops())


def coreset_tables(plan: Plan, unpooled_argsort: torch.Tensor, pooled_argsort: torch.Tensor):
    """(kept_tok, dropped_tok, unpool_src) int32 token tables from a MatchingResults pair
    (the index arithmetic of coreset_select.py:159-166)."""
    if not unpooled_argsort.is_cuda:
        raise L.VortaB200Error("coreset_tables needs CUDA tensors: vorta_b200 has no CPU path")
    un = unpooled_argsort.to(torch.int64).contiguous()
    po = pooled_argsort.to(torch.int64).contiguous()
    B, H = un.shape[:2]
    dev = un.device
    kept = torch.empty((B, H, plan.coreset_len + plan.text_len), dtype=torch.int32, device=dev)
    drop = torch.empty((B, H, plan.num_groups, max(plan.num_pooled, 1)), dtype=torch.int32, device=dev)
    src = torch.empty((B, H, plan.seq_len), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.lib().vb_coreset_tables(plan.handle, un.data_ptr(), po.data_ptr(), B, H, kept.data_ptr(),
                                          drop.data_ptr(), src.data_ptr(), _stream_ptr(dev)))
    return kept, drop[..., :plan.num_pooled], src


def attn_dense(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(Q K^T / sqrt(128)) V with independent query / key lengths (wan.py:142-144), (B, H, N, 128) views."""
    for name, t in (("q", q), ("k", k), ("v", v)):
        _require_cuda_bf16(name, t)
    B, H, Nq, D = q.shape
    Nk = k.shape[2]
    if k.shape != v.shape or k.shape[:2] != q.shape[:2]:
        raise ValueError(f"k and v must be (B={B}, H={H}, Nk, {D}) alike, got {tuple(k.shape)} and {tuple(v.shape)}")
    if out is None:
        out = torch.empty((B, Nq, H, D), dtype=q.dtype, device=q.device).transpose(1, 2)
    else:
        _require_cuda_bf16("out", out)
        if out.shape != q.shape:
            raise ValueError(f"out must have q's shape {tuple(q.shape)}, got {tuple(out.shape)}")
    i64x3 = C.c_int64 * 3
    with torch.cuda.device(q.device):
        L.check(L.lib().vb_attn_dense(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                      i64x3(*q.stride()[:3]), i64x3(*k.stride()[:3]), i64x3(*v.stride()[:3]),
                                      i64x3(*out.stride()[:3]), B, H, Nq, Nk, _stream_ptr(q.device)))
    return out


def timing_enable(on: bool) -> None:
    L.lib().vb_timing_enable(1 if on else 0)


def timing_collect() -> Tuple[float, int, float]:
    """(summed attention-kernel ms, launches, algorithmic FLOPs) since the last collect; waits for the events."""
    ms, n, fl = C.c_double(), C.c_int64(), C.c_double()
    L.check(L.lib().vb_timing_collect(C.byref(ms), C.byref(n), C.byref(fl)))
    return float(ms.value), int(n.value), float(fl.value)


def timing_collect_kinds():
    """Per caller: {"routed": (ms, launches, flops), "dense": (...)} — vb_attn_fwd launches (a layer's routed
    self-attention, all branches in one grid) and vb_attn_dense launches (cross attention etc.) of the same kernel."""
    ms, n, fl = (C.c_double * 2)(), (C.c_int64 * 2)(), (C.c_double * 2)()
    L.check(L.lib().vb_timing_collect_kinds(ms, n, fl))
    return {"routed": (float(ms[0]), int(n[0]), float(fl[0])), "dense": (float(ms[1]), int(n[1]), float(fl[1]))}


# ---------------------------------------------------------------------------------------------------------
# fused elementwise kernels of the DiT block around the path (SURVEY.md section 8f rows 1-2)
# ---------------------------------------------------------------------------------------------------------
def _rows(x: torch.Tensor):
    if not x.is_cuda:
        raise L.VortaB200Error("block kernels need CUDA tensors: vorta_b200 has no CPU path")
    if x.dtype != torch.bfloat16 or x.dim() != 3 or not x.is_contiguous():
        raise ValueError("block kernels need contiguous bf16 tensors of shape (B, S, dim)")
    return x.shape[0] * x.shape[1], x.shape[2], x.shape[1]


def _contig(x: torch.Tensor) -> torch.Tensor:
    return x if x.is_contiguous() else x.contiguous()


def _f32(t: Optional[torch.Tensor]):
    if t is None:
        return None
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.float().contiguous()
    return t


def ln_modulate(x: torch.Tensor, weight: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
                scale: Optional[torch.Tensor] = None, shift: Optional[torch.Tensor] = None,
                eps: float = 1e-6) -> torch.Tensor:
    """(LayerNorm(x) [* weight + bias]) [* (1 + scale) + shift] in fp32, one pass (modeling_wan.py:205-206)."""
    x = _contig(x)
    rows, dim, per_batch = _rows(x)
    weight, bias, scale, shift = _f32(weight), _f32(bias), _f32(scale), _f32(shift)
    out = torch.empty_like(x)
    p = lambda t: t.data_ptr() if t is not None else None
    with torch.cuda.device(x.device):
        L.check(L.lib().vb_block_ln_modulate(x.data_ptr(), p(weight), p(bias), p(scale), p(shift), out.data_ptr(), rows,
                                             dim, per_batch, float(eps), _stream_ptr(x.device)))
    return out


def gate_residual(x: torch.Tensor, y: torch.Tensor, gate: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x + y * gate in fp32, one pass (modeling_wan.py:225, 238); gate (B, dim) fp32 or None."""
    x = _contig(x)
    rows, dim, per_batch = _rows(x)
    if y.shape != x.shape:
        raise ValueError("gate_residual: shape mismatch")
    if not y.is_contiguous():
        y = y.contiguous()
    gate = _f32(gate)
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        L.check(L.lib().vb_block_gate_residual(x.data_ptr(), y.data_ptr(), gate.data_ptr() if gate is not None else None,
                                               out.data_ptr(), rows, dim, per_batch, _stream_ptr(x.device)))
    return out


def rmsnorm_rope(x: torch.Tensor, weight: torch.Tensor, eps: float, cos: Optional[torch.Tensor] = None,
                 sin: Optional[torch.Tensor] = None) -> torch.Tensor:
    """RMSNorm across heads * weight, then RoPE per 128-wide head (wan.py:85-100); cos / sin fp32 (S, 64)."""
    x = _contig(x)
    rows, dim, per_batch = _rows(x)
    w = weight if weight.dtype == torch.bfloat16 and weight.is_contiguous() else weight.to(torch.bfloat16).contiguous()
    out = torch.empty_like(x)
    if cos is not None and (tuple(cos.shape) != (per_batch, HEAD_DIM // 2) or cos.dtype != torch.float32):
        raise ValueError(f"cos / sin tables must be fp32 ({per_batch}, {HEAD_DIM // 2}), got {tuple(cos.shape)}")
    with torch.cuda.device(x.device):
        L.check(L.lib().vb_block_rmsnorm_rope(x.data_ptr(), w.data_ptr(), cos.data_ptr() if cos is not None else None,
                                              sin.data_ptr() if sin is not None else None, out.data_ptr(), rows, dim,
                                              per_batch, float(eps), _stream_ptr(x.device)))
    return out


def headnorm_rope(x: torch.Tensor, weight: Optional[torch.Tensor], eps: float, heads: int,
                  cos: Optional[torch.Tensor] = None, sin: Optional[torch.Tensor] = None,
                  rope_rows: Optional[int] = None, out: Optional[torch.Tensor] = None, dst_row0: int = 0
                  ) -> torch.Tensor:
    """Per-head RMSNorm * weight (128), then RoPE on the first ``rope_rows`` rows, written into rows
    [dst_row0, dst_row0 + rows) of ``out`` (B, dst_rows, heads * 128) — hunyuan.py:62-134 in one pass.
    x: (B, rows, heads * 128) bf16 contiguous; cos / sin fp32 (>= rope_rows, 64).  ``out`` defaults to in place."""
    if not x.is_cuda:
        raise L.VortaB200Error("block kernels need CUDA tensors: vorta_b200 has no CPU path")
    if x.dtype != torch.bfloat16 or x.dim() != 3 or not x.is_contiguous() or x.shape[2] != heads * HEAD_DIM:
        raise ValueError(f"headnorm_rope needs a contiguous bf16 (B, rows, {heads * HEAD_DIM}) tensor, got {tuple(x.shape)}")
    B, rows, _ = x.shape
    if out is None:
        out = x
    if (out.dtype != torch.bfloat16 or out.dim() != 3 or not out.is_contiguous() or out.shape[0] != B
            or out.shape[2] != x.shape[2]):
        raise ValueError("headnorm_rope: out must be a contiguous bf16 (B, dst_rows, heads * 128) tensor")
    w = None
    if weight is not None:
        w = weight if weight.dtype == torch.bfloat16 and weight.is_contiguous() else weight.to(torch.bfloat16).contiguous()
        if w.numel() != HEAD_DIM:
            raise ValueError(f"per-head RMSNorm weight must have {HEAD_DIM} entries, got {w.numel()}")
    n_rope = 0
    if cos is not None:
        n_rope = rows if rope_rows is None else int(rope_rows)
        if cos.dtype != torch.float32 or sin.dtype != torch.float32 or cos.shape[-1] != HEAD_DIM // 2 or \
                cos.shape[0] < n_rope or not cos.is_contiguous() or not sin.is_contiguous():
            raise ValueError(f"cos / sin tables must be contiguous fp32 (>= {n_rope}, {HEAD_DIM // 2})")
    with torch.cuda.device(x.device):
        L.check(L.lib().vb_block_headnorm_rope(x.data_ptr(), w.data_ptr() if w is not None else None,
                                               cos.data_ptr() if cos is not None else None,
                                               sin.data_ptr() if cos is not None else None, out.data_ptr(), B, rows,
                                               heads, n_rope, out.shape[1], int(dst_row0), float(eps),
                                               _stream_ptr(x.device)))
    return out
