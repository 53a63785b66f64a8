"""Plan tables built by the C library (host integer code) against the golden vectors and the oracle — CPU only."""
import numpy as np
import pytest
import torch

from oracle import vorta_oracle as O
from vorta_b200 import _lib as L
from vorta_b200 import ops
from vorta_b200.attention import create_sliding_tile_attn_mask_func, get_group_info
from vorta_b200.patch import prepare_hunyuan_self_attn_kwargs, prepare_wan_self_attn_kwargs, wan_pixel2token


def test_group_tables_bit_exact(golden):
    for rec in golden("group_info.pt"):
        info = get_group_info(rec["latent"], rec["window"], rec["rate"])
        assert info.num_unpooled_tokens_per_group == rec["n_unpooled"]
        assert info.center_indices.dtype == torch.int64 and info.margin_indices.dtype == torch.int64
        assert (tuple(info.center_indices.shape), tuple(info.margin_indices.shape)) == rec["shape"]
        assert int(info.center_indices.sum()) == rec["center_sum"]
        assert int(info.margin_indices.sum()) == rec["margin_sum"]
        assert torch.equal(info.center_indices[:16], rec["center_head"])
        assert torch.equal(info.margin_indices[-4:], rec["margin_tail"])
        if rec["center"] is not None:
            assert torch.equal(info.center_indices, rec["center"])
            assert torch.equal(info.margin_indices, rec["margin"])


def _mask_from_plan(plan, lat, tile, tl, tv):
    """Expand the plan's run tables back to a dense tile-major mask (test-side only)."""
    S = plan.seq_len
    tau = plan.tile_tokens
    runs = plan.export(L.EXPORT_SLIDING_RUNS).reshape(-1, 2)
    wins = plan.export(L.EXPORT_TILE_WINDOW).reshape(-1, 6)
    nt = [lat[d] // tile[d] for d in range(3)]
    n = S + tl
    mask = torch.zeros(n, n, dtype=torch.bool)
    for t in range(wins.shape[0]):
        lo, hi = wins[t, :3], wins[t, 3:]
        for a in range(lo[0], hi[0] + 1):
            for b in range(lo[1], hi[1] + 1):
                k0 = ((a * nt[1] + b) * nt[2] + lo[2]) * tau
                k1 = ((a * nt[1] + b) * nt[2] + hi[2] + 1) * tau
                mask[t * tau:(t + 1) * tau, k0:k1] = True
        mask[t * tau:(t + 1) * tau, S:S + tv] = True
    mask[S:S + tv, :S + tv] = True
    return mask, runs


def test_sliding_schedule_equals_reference_mask(golden):
    for rec in golden("tile_mask.pt"):
        lat, win, tile, tl, tv = rec["latent"], rec["window"], rec["tile"], rec["text_len"], rec["text_valid"]
        plan = ops.Plan(lat, tile, win, (1, 1, 1), n_unpooled=0, text_len=tl, text_valid=tv)
        tile_map = plan.export(L.EXPORT_TILE_MAP)
        assert np.array_equal(tile_map[:plan.seq_len], rec["tile_perm"].numpy())
        assert np.array_equal(tile_map[plan.seq_len:], np.arange(plan.seq_len, plan.seq_len + tl))
        mask, runs = _mask_from_plan(plan, lat, tile, tl, tv)
        n = mask.shape[0]
        ref = torch.from_numpy(np.unpackbits(rec["mask_bits"].numpy())[:n * n].reshape(n, n).astype(bool))
        assert torch.equal(mask, ref)
        assert plan.query(L.PLAN_KEYS_PER_QUERY) + tv == rec["keys_q0"]
        assert np.array_equal(plan.export(L.EXPORT_TILE_WINDOW).reshape(-1, 6), O.tile_windows(lat, win, tile))
        # the run table covers exactly the allowed keys of every query tile
        assert (runs[:, 1] > 0).all()


def _window_groups(plan):
    """Window groups in order of first appearance: (window, [tile ids])."""
    wins = plan.export(L.EXPORT_TILE_WINDOW).reshape(-1, 6)
    order, members = [], {}
    for t, w in enumerate(map(tuple, wins.tolist())):
        if w not in members:
            members[w] = []
            order.append(w)
        members[w].append(t)
    return [(w, members[w]) for w in order]


def test_run_table_expands_to_mask_rows():
    lat, win, tile = (4, 8, 12), (3, 3, 3), (2, 4, 4)
    plan = ops.Plan(lat, tile, win, (1, 1, 1), n_unpooled=0)
    runs = plan.export(L.EXPORT_SLIDING_RUNS).reshape(-1, 2)
    mask = O.sliding_tile_mask(lat, win, tile)
    tau = plan.tile_tokens
    # window groups appear in order of their first tile, each with its own consecutive set of runs whose union is
    # the mask row of EVERY tile of the group
    idx = 0
    for _, tiles in _window_groups(plan):
        row = mask[tiles[0] * tau]
        want = int(row.sum())
        got = torch.zeros_like(row)
        while want > int(got.sum()):
            s, n = runs[idx]
            assert not got[s:s + n].any()
            got[s:s + n] = True
            idx += 1
        for t in tiles:
            assert torch.equal(got, mask[t * tau]) and torch.equal(got, mask[(t + 1) * tau - 1])
    assert idx == runs.shape[0]


def test_sliding_query_map_is_window_group_order():
    """VB_EXPORT_SLIDING_QUERY_MAP: a permutation of the raster tokens that lists the tiles window group by window
    group (tiles whose clamped windows coincide are neighbours), tokens inside a tile in tile.py's order."""
    for lat, tile, win, tl in [((21, 45, 80), (3, 9, 16), (3, 3, 3), 0), ((21, 30, 52), (3, 10, 4), (3, 3, 3), 0),
                               ((4, 8, 8), (2, 4, 4), (3, 3, 3), 16), ((6, 6, 8), (1, 3, 4), (3, 1, 3), 0),
                               ((4, 4, 4), (2, 2, 2), (5, 5, 5), 0)]:
        plan = ops.Plan(lat, tile, win, (1, 1, 1), n_unpooled=0, text_len=tl, text_valid=tl)
        S, tau = plan.seq_len, plan.tile_tokens
        qmap = plan.export(L.EXPORT_SLIDING_QUERY_MAP)
        tmap = plan.export(L.EXPORT_TILE_MAP)
        assert qmap.shape[0] == S + tl and np.array_equal(np.sort(qmap), np.arange(S + tl))
        assert np.array_equal(qmap[S:], np.arange(S, S + tl))
        want = np.concatenate([tmap[t * tau:(t + 1) * tau] for _, tiles in _window_groups(plan) for t in tiles])
        assert np.array_equal(qmap[:S], want)
    # Wan-14B: 45 distinct windows over 175 tiles -> 606 query slots of 128 rows instead of 700
    plan = ops.Plan((21, 45, 80), (3, 9, 16), (3, 3, 3), (1, 1, 1), n_unpooled=0)
    groups = _window_groups(plan)
    assert len(groups) == 45 and sum(len(t) for _, t in groups) == 175
    items = plan.export(L.EXPORT_SLIDING_ITEMS).reshape(-1, 12)
    assert int(items[:, 6].sum()) == sum(-(-len(t) * 432 // 128) for _, t in groups) == 606


def test_baseline_shapes_build():
    # BASELINE.json grids with the substitute hyper-parameters of SURVEY.md section 8d
    for lat, tile, lw in [((21, 30, 52), (3, 10, 4), (3, 3, 2)), ((21, 45, 80), (3, 9, 16), (3, 3, 2)),
                          ((20, 45, 80), (5, 9, 8), (2, 3, 2)), ((33, 45, 80), (3, 9, 16), (3, 3, 2))]:
        plan = ops.Plan(lat, tile, (3, 3, 3), lw, 0.5)
        S = lat[0] * lat[1] * lat[2]
        assert plan.seq_len == S and plan.coreset_len == S // 2
        assert plan.query(L.PLAN_KEYS_PER_QUERY) == 27 * plan.tile_tokens
        for e in range(3):
            ref = O.branch_flops(e, lat, (3, 3, 3), tile, lw, 0.5)
            assert abs(plan.flops_per_head(e) - ref) / ref < 1e-12


def test_prepare_kwargs_mirror_reference_keys():
    kw = dict(latent_shape=(4, 6, 8), window_size=(3, 3, 3), tile_size=(2, 3, 4), lowres_window_size=(2, 3, 2),
              lowres_reduction_rate=0.5)
    out = prepare_wan_self_attn_kwargs(dict(kw), torch.device("cpu"), tau_sparse=0.3)
    assert set(out) == {"latent_shape", "window_size", "tile_size", "lowres_group_info", "flex_attn_mask_func",
                        "tau_sparse"}
    out = prepare_hunyuan_self_attn_kwargs(dict(kw), torch.device("cpu"))
    assert set(out) == {"latent_shape", "window_size", "tile_size", "lowres_group_info"}
    assert wan_pixel2token((77, 720, 1280)) == (20, 45, 80)
    assert wan_pixel2token((81, 480, 832)) == (21, 30, 52)
    with pytest.raises(ValueError):
        wan_pixel2token((78, 720, 1280))
    sched = create_sliding_tile_attn_mask_func((4, 6, 8), (3, 3, 3), (2, 3, 4), 0, 0)
    assert sched.tile_windows().shape == (8, 6)


def test_balance_heads_is_a_valid_and_better_placement():
    """Cost-balanced Ulysses head placement (vorta_b200/ulysses/balance.py): a permutation with H/P heads per rank,
    never worse than the reference's contiguous chunks, deterministic, identity -> None."""
    import random
    from vorta_b200.ulysses import balance_heads
    costs = [2.93, 0.73, 0.45]          # Wan-14B 720p TFLOP per head: full / coreset / sliding (SURVEY.md 8d)
    rng = random.Random(7)
    worse = 0
    for world in (2, 4, 8):
        for _ in range(200):
            H = 40
            branch = [rng.choice([0, 1, 2]) for _ in range(H)]
            hp = H // world
            head_at = balance_heads(branch, costs, world)
            contiguous = max(sum(costs[e] for e in branch[r * hp:(r + 1) * hp]) for r in range(world))
            if head_at is None:
                continue
            assert sorted(head_at) == list(range(H))
            assert head_at == balance_heads(list(branch), costs, world)
            for r in range(world):
                chunk = head_at[r * hp:(r + 1) * hp]
                assert chunk == sorted(chunk)
            load = max(sum(costs[branch[h]] for h in head_at[r * hp:(r + 1) * hp]) for r in range(world))
            assert load < contiguous
            ideal = sum(costs[e] for e in branch) / world
            worse += load > 1.35 * ideal
    assert worse == 0                                      # LPT stays close to the ideal split on this cost mix
    assert balance_heads([0] * 8, costs, 4) is None        # uniform routing: contiguous is already optimal
    assert balance_heads([0, 1, 2], costs, 1) is None
    assert balance_heads([0, 1, 2], costs, 2) is None      # heads not divisible: left to the caller's error path


def test_flow_match_euler_scheduler_cpu():
    """Scheduler restatement used by the denoise loops: sigmas fall from 1 to 0, timesteps = 1000 sigma, an Euler step
    along a constant velocity field integrates exactly to x0 - v."""
    from vorta_b200.patch.pipeline import FlowMatchEulerScheduler
    for shift in (1.0, 3.0, 7.0):
        sch = FlowMatchEulerScheduler(shift=shift)
        sch.set_timesteps(10)
        assert sch.timesteps.shape == (10,) and sch.sigmas.shape == (11,)
        assert abs(float(sch.sigmas[0]) - 1.0) < 1e-6 and float(sch.sigmas[-1]) == 0.0
        assert bool((sch.sigmas[1:] < sch.sigmas[:-1]).all())
        assert torch.allclose(sch.timesteps, sch.sigmas[:-1] * 1000)
        x, v = torch.full((2, 3), 5.0), torch.full((2, 3), 2.0)
        for t in sch.timesteps:
            x = sch.step(v, t, x)[0]
        assert torch.allclose(x, torch.full((2, 3), 3.0), atol=1e-5)


def test_top1_routing_matches_reference_rule():
    """wan.py:396-400: top-1 expert of the FIRST sample per head; below tau_sparse -> full attention (0)."""
    from vorta_b200.attention.wan import _top1_branches
    score = torch.tensor([[[0.5, 0.3, 0.2], [0.2, 0.45, 0.35], [0.1, 0.2, 0.7], [0.34, 0.33, 0.33]],
                          [[0.0, 1.0, 0.0]] * 4])                       # second sample is ignored
    assert _top1_branches(score, 0.3) == [0, 1, 2, 0]
    assert _top1_branches(score, 0.5) == [0, 0, 2, 0]                    # 0.45 < tau -> full
    assert _top1_branches(score, None) == [0, 1, 2, 0]
    assert _top1_branches(score, 0.75) == [0, 0, 0, 0]


def test_local_heads_follow_the_head_table():
    from vorta_b200.ulysses import SP_STATE, local_heads
    vals = list("abcdefgh")
    assert local_heads(vals, 8) == vals                                  # SP disabled: untouched
    SP_STATE._enabled, SP_STATE._sp_size, old_rank = True, 4, SP_STATE.__dict__.get("_group_local_rank")
    try:
        SP_STATE._group_local_rank = 2
        if SP_STATE.group_local_rank != 2:
            pytest.skip("SP_STATE does not expose a settable local rank")
        assert local_heads(vals, 8) == ["e", "f"]
        assert local_heads(vals, 8, head_at=[0, 7, 1, 6, 2, 5, 3, 4]) == ["c", "f"]
    finally:
        SP_STATE._enabled, SP_STATE._sp_size = False, 1
        if old_rank is not None:
            SP_STATE._group_local_rank = old_rank


def test_routed_output_container_behaves_like_base_output():
    """vorta/patch/outputs.py: attribute, key and index access; to_tuple skips None fields (diffusers BaseOutput)."""
    from vorta_b200.patch import RoutedTransformerModelOutput, VideoPipelineOutput
    x = torch.zeros(2)
    out = RoutedTransformerModelOutput(sample=x, routing_scores=[])
    assert out.sample is x and out["sample"] is x and out[0] is x
    assert out.to_tuple() == (x, []) and out.reg_loss is None
    full = RoutedTransformerModelOutput(x, torch.ones(()), torch.ones(()), torch.ones(()), [x])
    assert len(full.to_tuple()) == 5 and full[4] == [x]
    vid = VideoPipelineOutput(frames=x)
    assert vid.frames is x and vid.to_tuple() == (x,)


def test_router_checkpoint_roundtrip_with_reference_key_names(tmp_path):
    """``router.pt`` of the reference (vorta/train/checkpoint.py:31-43 saves, :63-74 loads): the transformer's own
    state-dict keys ``blocks.{i}.router.linear.{weight,bias}``.  Loading must set exactly the routers, leave every
    other parameter alone and drop keys the model does not have (``k in full_state_dict``), e.g. a checkpoint trained
    on a deeper model — not everything whose name merely contains "router"."""
    from vorta_b200.dit import WanDiT
    from vorta_b200.patch import apply_vorta_transformer, load_router_checkpoint
    dev = torch.device("cpu")
    model = apply_vorta_transformer(WanDiT.build("wan-contract-test", dev, torch.float32, seed=0))
    n_blocks = len(model.blocks)
    keys = [k for k in model.state_dict() if ".router." in k]
    assert sorted(keys) == sorted(f"blocks.{i}.router.linear.{p}" for i in range(n_blocks) for p in ("weight", "bias"))
    g = torch.Generator().manual_seed(3)
    ckpt = {k: torch.randn(model.state_dict()[k].shape, generator=g) for k in keys}
    ckpt[f"blocks.{n_blocks}.router.linear.weight"] = torch.zeros(3, 3)         # block the model does not have
    ckpt["router_ema.decay"] = torch.tensor(0.5)                                 # contains "router", not a model key
    path = tmp_path / "router.pt"
    torch.save(ckpt, path)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    load_router_checkpoint(path, model)
    after = model.state_dict()
    for k in after:
        if k in keys:
            assert torch.equal(after[k], ckpt[k])
        else:
            assert torch.equal(after[k], before[k])
    # a second model built through the install entry point with checkpoint_file= ends up with the same routers
    model2 = apply_vorta_transformer(WanDiT.build("wan-contract-test", dev, torch.float32, seed=1), checkpoint_file=path)
    for k in keys:
        assert torch.equal(model2.state_dict()[k], ckpt[k])


@pytest.mark.parametrize("lat,tile,win,tl,tv", [
    ((21, 30, 52), (3, 10, 4), (3, 3, 3), 0, 0),      # Wan-1.3B: 120-token tiles -> every item is a split pair
    ((21, 45, 80), (3, 9, 16), (3, 3, 3), 0, 0),      # Wan-14B: 432-token tiles -> two shared-run items per tile
    ((20, 45, 80), (5, 9, 8), (3, 3, 3), 0, 0),       # reference-native: 360 = 256 + 104 -> one shared + one single item
    ((4, 8, 8), (2, 4, 4), (3, 3, 3), 16, 11),        # text segment: text queries are their own items
    ((6, 6, 8), (1, 3, 4), (3, 1, 3), 0, 0),          # tiny tiles (12 tokens), odd tile count
])
def test_sliding_work_items_cover_every_query_once_with_its_window(lat, tile, win, tl, tv):
    """The work items of the persistent attention kernel (vb_attn.cu): every query position of the sliding branch
    (VB_EXPORT_SLIDING_QUERY_MAP order) is in exactly one 128-row slot; the run list of its slot is the window of the
    tile that token belongs to (bit-exact against the oracle's dense mask); items that pair two slots with different
    windows ("split") walk the same number of key blocks; items are ordered longest first."""
    plan = ops.Plan(lat, tile, win, (1, 1, 1), 0.5, text_len=tl, text_valid=tv, n_unpooled=0)
    items = plan.export(L.EXPORT_SLIDING_ITEMS).reshape(-1, 12)
    runs = plan.export(L.EXPORT_SLIDING_RUNS).reshape(-1, 2)
    qmap = plan.export(L.EXPORT_SLIDING_QUERY_MAP)
    S, tau = plan.seq_len, plan.tile_tokens
    nt = [lat[d] // tile[d] for d in range(3)]
    wins = O.tile_windows(lat, win, tile)
    dense = O.sliding_tile_mask(lat, win, tile, tl, tv) if S <= 4096 else None     # tile-major index space
    tile_pos = np.empty(S + tl, dtype=np.int64)      # raster token -> tile-major position
    tile_pos[plan.export(L.EXPORT_TILE_MAP)] = np.arange(S + tl)

    def merged(intervals):
        out = []
        for a, b in sorted(intervals):
            if out and out[-1][1] == a:
                out[-1][1] = b
            else:
                out.append([a, b])
        return out

    def expected_keys(pos):                            # pos: tile-major position of the query
        if pos >= S:                                   # a valid text query sees every non-pad key
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
            assert sum((e - st + 127) // 128 for st, e in mine) == nblk
            # every sliding tile the slot touches (its rows may span several tiles of one window group)
            rows = sorted({q0, q0 + qr - 1} | {r for r in range(q0, q0 + qr) if r < S and r % tau == 0})
            for r in rows:
                pos = int(tile_pos[qmap[r]])
                assert merged(mine) == expected_keys(pos), (q0, qr, r)
                if dense is not None:
                    keys = torch.zeros(S + tl, dtype=torch.bool)
                    for st, e in mine:
                        keys[st:e] = True
                    assert torch.equal(keys, dense[pos])
        cost.append(nblk * nq)
    assert (seen == 1).all()
    assert cost == sorted(cost, reverse=True)
    n_slots = sum(it[6] for it in items.tolist())
    groups = _window_groups(plan)
    assert n_slots == sum(-(-len(t) * tau // 128) for _, t in groups) + (-(-tv // 128) if tv else 0)
    assert n_slots <= plan.num_tiles * -(-tau // 128) + (-(-tv // 128) if tv else 0)


def test_placement_with_query_half_units():
    """balance.place_units: deterministic; every head is held exactly once — whole, or as a lower and an upper query
    half (full-attention heads only); at most `slots` units per rank; never worse than the whole-head placement, and
    clearly better where a rank holds only a few heads (HunyuanVideo: 24 heads on 8 ranks)."""
    import random
    from vorta_b200.ulysses import balance
    costs = [6.5, 1.8, 1.25]
    rnd = random.Random(3)
    gain = []
    for H, P in ((40, 8), (24, 8), (40, 4), (12, 2), (24, 4)):
        slots = balance.max_slots(H, P)
        for _ in range(10):
            branch = [rnd.choice([0, 1, 2]) for _ in range(H)]
            placed = balance.place_units(branch, costs, P, slots)
            assert placed == balance.place_units(list(branch), costs, P, slots)
            assert len(placed) == P and max(len(u) for u in placed) <= slots
            seen = {}
            for units in placed:
                for h, part in units:
                    seen.setdefault(h, []).append(part)
            assert sorted(seen) == list(range(H))
            for h, parts in seen.items():
                if parts == [balance.WHOLE]:
                    continue
                n = balance.part_kn(parts[0])[1]           # a split head: every part k of n exactly once
                assert branch[h] == 0 and n == 2
                assert sorted(parts) == [balance.part_code(k, n) for k in range(n)]

            def load(p):
                return max(sum(costs[branch[h]] * (1.0 if part == balance.WHOLE else 1.03 / balance.part_kn(part)[1])
                               for h, part in u) for u in p)
            whole = balance.place_units(branch, costs, P, slots, allow_split=False)
            assert all(part == balance.WHOLE for u in whole for _, part in u)
            assert load(placed) <= load(whole) * (1 + 1e-9)
            if (H, P) == (24, 8):
                gain.append(load(whole) / load(placed))
    assert max(gain) > 1.04 and min(gain) >= 1.0


_PLACEMENT_PLANS = {          # the bench workloads' geometries (bench.py WORKLOADS)
    "wan14": dict(latent_shape=(21, 45, 80), tile_size=(3, 9, 16), window_size=(3, 3, 3),
                  lowres_window_size=(3, 3, 2)),
    "hunyuan": dict(latent_shape=(33, 45, 80), tile_size=(3, 9, 16), window_size=(3, 3, 3),
                    lowres_window_size=(3, 3, 2), text_len=256, text_valid=64),
}


def test_ulysses_placements_match_recorded_answers():
    """Which rank computes which head, pinned: the NCCL head table (balance_heads), the peer-memory unit table
    (layer_placement) and every rank's (branch ids, out_heads) for vb_attn_fwd, recorded from the placement code before
    the two processors shared one dispatch.  Bench routing (7h+1)%3 and three seeded random routings; Wan-14B (40 heads,
    P = 2, 4, 8) and HunyuanVideo (24 heads, P = 8) with the branch costs of the real plans."""
    import json
    import os
    from vorta_b200.ulysses import balance
    from vorta_b200.ulysses.routed import local_units
    with open(os.path.join(os.path.dirname(__file__), "golden", "ulysses_placements.json")) as f:
        cases = json.load(f)["cases"]
    plans = {name: ops.Plan(**geometry) for name, geometry in _PLACEMENT_PLANS.items()}
    for c in cases:
        plan, branch, P, slots = plans[c["workload"]], c["branch"], c["world"], c["slots"]
        what = (c["workload"], P, c["routing"])
        assert balance.branch_costs(plan) == c["costs"], what
        assert balance.max_slots(len(branch), P) == slots, what
        assert balance.balance_heads(branch, c["costs"], P) == c["head_at"], what
        placement = balance.layer_placement(branch, plan, P, slots)
        assert [[list(u) for u in units] for units in placement] == c["placement"], what
        for r, want in enumerate(c["local_units"]):
            assert local_units(placement, r, branch, slots) == (want["ids"], want["out_heads"]), (what, r)
