"""Cost-balanced head placement for the Ulysses exchange (SURVEY.md section 8e).

The reference gives rank r the contiguous heads [r*H/P, (r+1)*H/P) (vorta/ulysses/utils.py:60-66).  With routed
attention the heads of one layer differ in cost by ~6x (full : coreset : sliding), every rank waits for the slowest
one at the "out" exchange, and the routing of the whole step is known before the first block runs — so the host
picks, per layer, which H/P heads each rank receives.  The choice only changes slot numbers inside the exchange
buffers (``head_at`` of ``vb_ulysses_*``; ``out_heads`` of ``vb_attn_fwd``): no extra bytes move, and results are
bit-identical to the contiguous placement because heads are independent.

Every placement is deterministic and depends only on (branch ids, costs, P): every rank derives the same table
from its own copy of the routing decisions.  ``balance_heads`` places whole heads, H/P per rank, for the NCCL
exchange; ``layer_placement`` places work units (whole heads and query halves) for the peer-memory exchange.  Both
run the same greedy ``_place``.
"""
from __future__ import annotations

import functools
from typing import List, Optional, Sequence

# measured time per algorithmic FLOP relative to the full branch, layout / selection passes included
# (profiles/r2e_perf_gather.log, r2m_perf_ab_final_kernel.log: full 1330-1370, coreset 1280-1290 incl. select + pool,
# sliding 1050-1070 kernel / 960-1050 incl. the tile-major pass, TFLOP/s at the Wan-14B geometry)
_BRANCH_OVERHEAD = (1.0, 1.06, 1.33)


def branch_costs(plan) -> List[float]:
    """Relative cost of one head of each branch for this geometry (algorithmic FLOPs x measured overhead)."""
    return [plan.flops_per_head(e) * _BRANCH_OVERHEAD[e] for e in range(3)]


def _head_costs(branch: Sequence[int], costs: Sequence[float]) -> List[float]:
    return [costs[e] if 0 <= e < len(costs) else 0.0 for e in branch]


def balance_heads(branch: Sequence[int], costs: Sequence[float], world: int) -> Optional[List[int]]:
    """Longest-processing-time placement of H heads on ``world`` ranks, H/world heads each.

    Returns ``head_at`` with ``head_at[r * H/P + i]`` = head held in slot i of rank r (ascending head order inside
    a rank), or None when the contiguous placement is already as good (identity tables skip the host work)."""
    H = len(branch)
    if world <= 1 or H % world != 0:
        return None
    hp = H // world
    branch, costs = tuple(int(e) for e in branch), tuple(float(c) for c in costs)
    held, load = _place(branch, costs, world, hp, False)
    cost = _head_costs(branch, costs)
    contiguous = max(sum(cost[r * hp:(r + 1) * hp]) for r in range(world))
    if load >= contiguous * (1.0 - 1e-9):
        return None
    return [h for units in held for h, _ in units]


# ------------------------------------------------------------------------------------------------------------------
# Placement in work units: whole heads, and query halves of full heads (peer-memory exchange only)
# ------------------------------------------------------------------------------------------------------------------
WHOLE = 0                              # part of a head a slot computes: all of its query work items, or


def part_code(k: int, n: int) -> int:
    """... part k of n equal parts of them (n >= 2), encoded like VB_BRANCH_FULL_PART minus 16."""
    return 8 * n + k


def part_kn(part: int):
    return part & 7, part >> 3


LOWER, UPPER = part_code(0, 2), part_code(1, 2)
_SPLIT_OVERHEAD = 1.03                 # a part costs a little more than its share (another copy of K / V crosses NVLink)


def split_enabled(world: int) -> bool:
    """Query-half units pay off when a rank holds only a few heads (3 at HunyuanVideo P = 8, 5 at Wan-14B P = 8: one full
    head is 20-40 % of a rank's layer time)."""
    return world >= 4


def max_slots(heads: int, world: int) -> int:
    """Head slots of a rank's receive buffer: room for an uneven placement and for split heads."""
    hp = heads // world
    return min(64, 2 * hp + (1 if hp < 4 else 0))


def place_units(branch: Sequence[int], costs: Sequence[float], world: int, slots: int, allow_split: bool = True
                ) -> List[List[tuple]]:
    """Greedy longest-processing-time placement of a layer's heads on ``world`` ranks with at most ``slots`` units per
    rank.  A unit is (head, part): a whole head, or — for full-attention heads, when that lowers the slowest rank's
    load — one query half of its work items (``LOWER`` / ``UPPER``; the halves may land on different ranks, each
    receives the head's K / V).
    Deterministic in (branch, costs, world, slots): every rank computes the same table.  Returns, per rank, its units
    in slot order.  Results are cached per routing (the same decisions recur across steps and CFG passes)."""
    placed, _ = _place(tuple(int(e) for e in branch), tuple(float(c) for c in costs), int(world), int(slots),
                       bool(allow_split))
    return [list(u) for u in placed]


def layer_placement(branch: Sequence[int], plan, world: int, slots: int) -> List[List[tuple]]:
    """Placement of one layer's heads for the peer exchange: cost-balanced units, with query halves of full heads from
    4 ranks up."""
    return place_units(branch, branch_costs(plan), world, slots, allow_split=split_enabled(world))


@functools.lru_cache(maxsize=4096)
def _place(branch: tuple, costs: tuple, world: int, slots: int, allow_split: bool):
    """-> (units of every rank, ascending, the largest load of a rank)."""
    H = len(branch)
    cost = _head_costs(branch, costs)

    def lpt(units):           # units sorted by (-cost, head, part)
        load = [0.0] * world
        count = [0] * world
        held = [[] for _ in range(world)]
        for c, h, part in units:
            best_r, best_l = -1, 0.0
            for r in range(world):
                if count[r] < slots and (best_r < 0 or load[r] < best_l):
                    best_r, best_l = r, load[r]
            if best_r < 0:
                return None, float("inf")
            held[best_r].append((h, part))
            count[best_r] += 1
            load[best_r] += c
        return held, max(load)

    def order(units):
        return sorted(units, key=lambda u: (-u[0], u[1], u[2]))

    whole = [(cost[h], h, WHOLE) for h in range(H)]
    best, best_load = lpt(order(whole))
    if allow_split:
        # try splitting the k most expensive full heads in halves (one split alone often does not lower the maximum:
        # several ranks tie at it); keep the candidate with the lowest maximum load, the fewest units among equals
        full = sorted((h for h in range(H) if branch[h] == 0), key=lambda h: (-cost[h], h))
        tried = sorted({k for k in (1, 2, 3, 4, 6, 8, 12, 16, 24, len(full)) if 1 <= k <= len(full)})
        for k in tried:
            chosen = set(full[:k])
            units = [u for u in whole if u[1] not in chosen]
            for h in full[:k]:
                share = cost[h] / 2 * _SPLIT_OVERHEAD
                units += [(share, h, LOWER), (share, h, UPPER)]
            placed, load = lpt(order(units))
            if placed is not None and load < best_load * (1.0 - 1e-3):
                best, best_load = placed, load
    if best is None:
        raise ValueError(f"{H} heads do not fit {world} ranks x {slots} slots")
    return tuple(tuple(sorted(u)) for u in best), best_load
