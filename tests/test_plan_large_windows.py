"""Plan tables of the large coreset windows (groups of more than 33 tokens) and of sliding windows that need more than
32 key runs per window group, against the pinned CPU oracle — CPU only.

The reference's goldens (tests/golden/) cover none of these geometries and none can be made without the reference's
code, so the oracle (held to those goldens by tests/test_oracle_golden.py) is the reference here: its
``get_group_info``, ``sliding_tile_mask`` and ``tile_windows`` are the reference's formulas for any window."""
import numpy as np
import pytest
import torch

from oracle import vorta_oracle as O
from vorta_b200 import _lib as L
from vorta_b200 import ops
from vorta_b200.attention import get_group_info

MAX_GROUP = 4843          # largest coreset group the selection kernel takes (12 B of shared memory per margin and warp)

# g in {36, 48, 64, 72, 128, 256}, one latent grid that all of them divide
GROUP_WINDOWS = [(1, 6, 6), (2, 4, 6), (4, 4, 4), (2, 6, 6), (2, 8, 8), (4, 8, 8)]
GROUP_LATENT = (8, 24, 24)


@pytest.mark.parametrize("lw", GROUP_WINDOWS, ids=lambda w: f"g{w[0] * w[1] * w[2]}")
def test_large_group_tables_equal_oracle(lw):
    """Centre slot and member order of every group, the pooled length S_c = G (1 + n_u) and the dropped count."""
    g = lw[0] * lw[1] * lw[2]
    ref = O.get_group_info(GROUP_LATENT, lw, 0.5)
    info = get_group_info(GROUP_LATENT, lw, 0.5)
    assert torch.equal(info.center_indices, ref.center_indices)
    assert torch.equal(info.margin_indices, ref.margin_indices)
    assert info.num_unpooled_tokens_per_group == ref.num_unpooled_tokens_per_group == int(g * 0.5) - 1
    plan = ops.Plan(GROUP_LATENT, (1, 1, 1), (1, 1, 1), lw, 0.5)
    G = int(np.prod(GROUP_LATENT)) // g
    assert plan.group_size == g and plan.num_groups == G
    assert plan.coreset_len == G * (1 + ref.num_unpooled_tokens_per_group)
    assert plan.num_pooled == g - 1 - ref.num_unpooled_tokens_per_group
    # every token is a centre or a margin of exactly one group
    allt = torch.cat([info.center_indices.flatten(), info.margin_indices.flatten()])
    assert torch.equal(allt.sort().values, torch.arange(plan.seq_len))


def test_largest_group_is_accepted_and_the_next_one_refused():
    lat = (29, 167, 1)                                      # 29 * 167 = 4843: one group over the whole grid
    plan = ops.Plan(lat, (1, 1, 1), (1, 1, 1), lat, 0.5)
    assert plan.group_size == MAX_GROUP and plan.num_groups == 1
    ref = O.get_group_info(lat, lat, 0.5)
    info = get_group_info(lat, lat, 0.5)
    assert torch.equal(info.center_indices, ref.center_indices) and torch.equal(info.margin_indices, ref.margin_indices)
    lat = (4, 7, 173)                                       # 4844 tokens
    with pytest.raises(RuntimeError, match=f"group of 4844 tokens exceeds the selection kernel's maximum of {MAX_GROUP}"):
        ops.Plan(lat, (1, 1, 1), (1, 1, 1), lat, 0.5)
    # the reference's own errors still come first
    with pytest.raises(ValueError, match="does not match low-res info"):
        ops.Plan((4, 7, 173), (1, 1, 1), (1, 1, 1), (3, 7, 173), 0.5)


# (latent, tile, window, text_len, text_valid): window groups with 33 to 101 key runs
LONG_RUNS = [
    ((11, 8, 8), (1, 2, 2), (11, 3, 3), 0, 0),            # window spans the whole t axis: 11 x 3 = 33 runs
    ((11, 8, 8), (1, 2, 2), (11, 3, 3), 16, 11),          # + the text run: 34
    ((33, 4, 4), (1, 2, 2), (11, 3, 1), 0, 0),            # window 11 along t over 33 one-frame tiles: 22 runs, and
    ((33, 4, 4), (1, 2, 2), (35, 5, 1), 0, 0),            # n < window on t and h (clamped to the grid): 66 runs
    ((9, 16, 4), (1, 4, 2), (9, 5, 1), 8, 8),             # 36 + 1 runs, every text row valid
    ((10, 20, 6), (1, 2, 2), (11, 11, 1), 8, 5),          # 10 x 10 + 1 = 101 runs, padded text rows
]


def _runs_per_group(items):
    return max(max(it[5], it[10]) for it in items.tolist())


@pytest.mark.parametrize("lat,tile,win,tl,tv", LONG_RUNS)
def test_long_run_schedule_equals_reference_mask(lat, tile, win, tl, tv):
    """The run table expanded to a dense tile-major mask equals the oracle's mask_mod bit for bit (as in
    test_sliding_schedule_equals_reference_mask), and the tile windows equal the oracle's."""
    plan = ops.Plan(lat, tile, win, (1, 1, 1), n_unpooled=0, text_len=tl, text_valid=tv)
    S, tau = plan.seq_len, plan.tile_tokens
    nt = [lat[d] // tile[d] for d in range(3)]
    wins = plan.export(L.EXPORT_TILE_WINDOW).reshape(-1, 6)
    assert np.array_equal(wins, O.tile_windows(lat, win, tile))
    runs = plan.export(L.EXPORT_SLIDING_RUNS).reshape(-1, 2)
    items = plan.export(L.EXPORT_SLIDING_ITEMS).reshape(-1, 12)
    n_max = _runs_per_group(items)
    assert n_max <= nt[0] * nt[1] + (1 if tv else 0)
    if win != (11, 3, 1):
        assert n_max > 32
    # every query row's mask row from the runs of the item that holds it
    qmap = plan.export(L.EXPORT_SLIDING_QUERY_MAP)
    tile_pos = np.empty(S + tl, dtype=np.int64)
    tile_pos[plan.export(L.EXPORT_TILE_MAP)] = np.arange(S + tl)
    mask = torch.zeros(S + tl, S + tl, dtype=torch.bool)
    for q0a, q0b, qra, qrb, rb, rc, nq, _, split, rb2, rc2, _ in items.tolist():
        slots = [(q0a, qra, rb, rc)] + ([(q0b, qrb, rb2, rc2) if split else (q0b, qrb, rb, rc)] if nq == 2 else [])
        for q0, qr, b, c in slots:
            pos = torch.from_numpy(tile_pos[qmap[q0:q0 + qr]])
            for st, ln in runs[b:b + c].tolist():
                assert ln > 0
                mask[pos, st:st + ln] = True
    ref = O.sliding_tile_mask(lat, win, tile, tl, tv)
    assert torch.equal(mask, ref)
    assert plan.query(L.PLAN_KEYS_PER_QUERY) + tv == int(ref[0].sum())


@pytest.mark.parametrize("lat,tile,win,tl,tv", LONG_RUNS)
def test_long_run_work_items_cover_every_query_once_with_its_window(lat, tile, win, tl, tv):
    """As test_sliding_work_items_cover_every_query_once_with_its_window: every query position is in exactly one
    128-row slot, its run list is its tile's window (merged intervals against the closed form), a slot's block count
    is that of its runs, split items pair equal block counts, and items are ordered longest first."""
    plan = ops.Plan(lat, tile, win, (1, 1, 1), n_unpooled=0, text_len=tl, text_valid=tv)
    items = plan.export(L.EXPORT_SLIDING_ITEMS).reshape(-1, 12)
    runs = plan.export(L.EXPORT_SLIDING_RUNS).reshape(-1, 2)
    qmap = plan.export(L.EXPORT_SLIDING_QUERY_MAP)
    S, tau = plan.seq_len, plan.tile_tokens
    nt = [lat[d] // tile[d] for d in range(3)]
    wins = O.tile_windows(lat, win, tile)
    tile_pos = np.empty(S + tl, dtype=np.int64)
    tile_pos[plan.export(L.EXPORT_TILE_MAP)] = np.arange(S + tl)

    def merged(intervals):
        out = []
        for a, b in sorted(intervals):
            if out and out[-1][1] == a:
                out[-1][1] = b
            else:
                out.append([a, b])
        return out

    def expected_keys(pos):
        if pos >= S:
            return [[0, S + tv]]
        lo, hi = wins[pos // tau, :3], wins[pos // tau, 3:]
        iv = [(((x * nt[1] + y) * nt[2] + lo[2]) * tau, ((x * nt[1] + y) * nt[2] + hi[2] + 1) * tau)
              for x in range(lo[0], hi[0] + 1) for y in range(lo[1], hi[1] + 1)]
        if tv:
            iv.append((S, S + tv))
        return merged(iv)

    seen = np.zeros(S + tv, dtype=np.int32)
    cost = []
    for q0a, q0b, qra, qrb, rb, rc, nq, nblk, split, rb2, rc2, _ in items.tolist():
        assert nq in (1, 2) and split in (0, 1) and (split == 0 or nq == 2)
        slots = [(q0a, qra, rb, rc)]
        if nq == 2:
            slots.append((q0b, qrb, rb2, rc2) if split else (q0b, qrb, rb, rc))
        for q0, qr, b, c in slots:
            assert 0 < qr <= 128
            seen[q0:q0 + qr] += 1
            mine = [(st, st + ln) for st, ln in runs[b:b + c].tolist()]
            assert sum((e - st + 127) // 128 for st, e in mine) == nblk      # 128-key blocks never cross a run
            for r in range(q0, q0 + qr):
                assert merged(mine) == expected_keys(int(tile_pos[qmap[r]])), (q0, qr, r)
        cost.append(nblk * nq)
    assert (seen == 1).all()
    assert cost == sorted(cost, reverse=True)


def test_long_run_plan_with_a_large_coreset_window():
    """Both lifted limits in one plan (the geometry of the GPU tests' Wan DiT step): a 48-token coreset window and
    sliding window groups of 36 runs."""
    lat, tile, win, lw = (12, 6, 8), (1, 2, 2), (13, 3, 3), (2, 3, 8)
    plan = ops.Plan(lat, tile, win, lw, 0.5)
    assert plan.group_size == 48 and plan.num_groups == 12 and plan.coreset_len == 12 * 24
    assert _runs_per_group(plan.export(L.EXPORT_SLIDING_ITEMS).reshape(-1, 12)) == 36
