"""Multi-GPU parity check, launched by torchrun (one rank per GPU): the Ulysses-parallel processors must reproduce
the single-GPU result (the N-GPU == 1-GPU contract of SURVEY.md section 5).  Prints one line per case; exits
non-zero on a mismatch.  Driven by tests/test_multigpu.py.

Usage: mgpu_check.py [MODE].  MODE "peer-split" forces query-half units at every world size, a MODE ending in
"-contiguous" keeps the reference's contiguous head chunks on the NCCL path; the exchange itself is chosen by the
VB_ULYSSES environment variable."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import fixtures as FX  # noqa: E402
from vorta_b200.attention import (HunyuanVideoFlashAttnProcessorTripleEval, WanAttnProcessorTripleEval,  # noqa: E402
                                  WanAttnProcessorTripleTrain, get_group_info)
from vorta_b200.ulysses import SP_STATE, all_gather, balance, peer  # noqa: E402


def main():
    mode = sys.argv[1] if len(sys.argv) > 1 else "peer"
    if mode == "peer-split":
        balance.split_enabled = lambda world: True
    if mode.endswith("-contiguous"):
        balance.balance_heads = lambda branch, costs, world: None
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ok = True

    def check(name, got, ref, tol=2e-2):
        nonlocal ok
        err = (got.float() - ref.float()).abs().max().item()
        scale = ref.float().abs().max().item()
        good = err <= tol * max(scale, 1.0)
        ok &= good
        if rank == 0:
            print(f"{name:40s} max_abs={err:.3e} (ref absmax {scale:.3e}) {'OK' if good else 'MISMATCH'}", flush=True)

    # ---------------- Wan: H = 4 * world heads so that every branch lands on every rank mix ----------------
    lat, tile, win, lw = (4, 6, 8), (2, 3, 4), (3, 3, 3), (2, 3, 2)
    S, H = 192, 4 * world
    attn = FX.FakeWanAttn(H, seed=5).to(dev, torch.bfloat16)
    hs = FX.det_tensor((1, S, H * 128), 6).to(dev, torch.bfloat16)
    rot = FX.wan_rotary(S, 7).to(dev)
    kw = dict(lowres_group_info=get_group_info(lat, lw, 0.5, device=dev), flex_attn_mask_func=None,
              window_size=win, tile_size=tile, latent_shape=lat)
    score = torch.softmax(FX.det_tensor((1, H, 3), 8, 4.0), -1).to(dev)
    ev, tr = WanAttnProcessorTripleEval(check_input=True), WanAttnProcessorTripleTrain(check_input=True)
    with torch.no_grad():
        ref_eval = ev(attn, hs, None, None, rot, tau_sparse=0.3, routing_score=score, **kw)
        ref_train = tr(attn, hs, None, None, rot, routing_score=score, **kw)
        ref_orig = ev(attn, hs, None, None, rot, tau_sparse=0.3, routing_score=score, use_original_attn=True, **kw)
        ctx = FX.det_tensor((1, 40, H * 128), 9).to(dev, torch.bfloat16)
        ref_cross = ev(attn, hs, ctx, None, None, tau_sparse=0.3, routing_score=score, **kw)
        # batch 2 (the reference's _all_to_all_4D takes any batch, utils.py:15-93): a second sample, its own scores
        hs2 = torch.cat([hs, FX.det_tensor((1, S, H * 128), 16).to(dev, torch.bfloat16)], dim=0)
        score2 = torch.cat([score, torch.softmax(FX.det_tensor((1, H, 3), 18, 4.0), -1).to(dev)], dim=0)
        ref_eval2 = ev(attn, hs2, None, None, rot, tau_sparse=0.3, routing_score=score2, **kw)
        ref_train2 = tr(attn, hs2, None, None, rot, routing_score=score2, **kw)
        ref_orig2 = ev(attn, hs2, None, None, rot, tau_sparse=0.3, routing_score=score2, use_original_attn=True, **kw)
    SP_STATE.setup_sp_group(world)
    s_loc = S // world
    mine = hs[:, rank * s_loc:(rank + 1) * s_loc].contiguous()
    with torch.no_grad():
        got = all_gather(ev(attn, mine, None, None, rot, tau_sparse=0.3, routing_score=score, **kw), dim=1)
        check("wan eval (top-1 routed)", got, ref_eval)
        got = all_gather(tr(attn, mine, None, None, rot, routing_score=score, **kw), dim=1)
        check("wan train (blend)", got, ref_train)
        got = all_gather(ev(attn, mine, None, None, rot, tau_sparse=0.3, routing_score=score, use_original_attn=True,
                            **kw), dim=1)
        check("wan original attention", got, ref_orig)
        got = all_gather(ev(attn, mine, ctx, None, None, tau_sparse=0.3, routing_score=score, **kw), dim=1)
        check("wan cross attention", got, ref_cross)
        mine2 = hs2[:, rank * s_loc:(rank + 1) * s_loc].contiguous()
        got = all_gather(ev(attn, mine2, None, None, rot, tau_sparse=0.3, routing_score=score2, **kw), dim=1)
        check("wan eval, batch 2", got, ref_eval2)
        got = all_gather(tr(attn, mine2, None, None, rot, routing_score=score2, **kw), dim=1)
        check("wan train (blend), batch 2", got, ref_train2)
        got = all_gather(ev(attn, mine2, None, None, rot, tau_sparse=0.3, routing_score=score2, use_original_attn=True,
                            **kw), dim=1)
        check("wan original attention, batch 2", got, ref_orig2)
    SP_STATE._enabled, SP_STATE._sp_size = False, 1        # single-GPU reference for the next case

    # ---------------- Wan dense baseline (apply_sp_flashattn_transformer) under SP: whole DiT step ----------------
    from vorta_b200.dit import WanDiT
    from vorta_b200.dit import wan as wan_mod
    from vorta_b200.patch import apply_sp_flashattn_transformer
    wan_mod.WAN_CONFIGS["mgpu"] = wan_mod.WanConfig(dim=H * 128, heads=H, ffn_dim=256, num_layers=2, text_dim=64)
    dense = apply_sp_flashattn_transformer(WanDiT.build("mgpu", dev, torch.bfloat16, seed=2))
    lat_in = FX.det_tensor((1, 16, lat[0], 2 * lat[1], 2 * lat[2]), 20).to(dev, torch.bfloat16)
    txt_in = FX.det_tensor((1, 12, 64), 21).to(dev, torch.bfloat16)
    ts_in = torch.tensor([300.0], device=dev)
    with torch.no_grad():
        ref_dense = dense(lat_in, ts_in, txt_in, return_dict=False)[0]
        SP_STATE._enabled, SP_STATE._sp_size = True, world
        got_dense = dense(lat_in, ts_in, txt_in, return_dict=False)[0]
        check("wan dense baseline DiT step (sp flashattn)", got_dense, ref_dense)
    SP_STATE._enabled, SP_STATE._sp_size = False, 1

    # ---------------- HunyuanVideo single-stream block with a padded text tail ----------------
    lat, tile, win, lw, TL, TV = (2, 8, 8), (1, 4, 4), (3, 3, 3), (2, 2, 2), 16, 11
    S = 128
    hattn = FX.FakeHunyuanAttn(H, dual=False, seed=11).to(dev, torch.bfloat16)
    hs = FX.det_tensor((1, S, H * 128), 12).to(dev, torch.bfloat16)
    ehs = FX.det_tensor((1, TL, H * 128), 13).to(dev, torch.bfloat16)
    mask = torch.zeros(1, 1, 1, S + TL, dtype=torch.bool, device=dev)
    mask[..., :S + TV] = True
    c, s = FX.hunyuan_rotary(S, 14)
    rope = (c.to(dev), s.to(dev))
    kw = dict(lowres_group_info=get_group_info(lat, lw, 0.5, device=dev), flex_attn_mask_func=None, window_size=win,
              tile_size=tile, latent_shape=lat)
    hev = HunyuanVideoFlashAttnProcessorTripleEval(check_input=True)
    with torch.no_grad():
        ref_v, ref_t = hev(hattn, hs, ehs, mask, rope, routing_score=score, tau_sparse=0.3, **kw)
    SP_STATE._enabled, SP_STATE._sp_size = True, world
    mine = hs[:, rank * (S // world):(rank + 1) * (S // world)].contiguous()
    with torch.no_grad():
        v, t = hev(hattn, mine, ehs, mask, rope, routing_score=score, tau_sparse=0.3, **kw)
        check("hunyuan single-stream eval (video)", all_gather(v, dim=1), ref_v)
        check("hunyuan single-stream eval (text)", t, ref_t)
    from vorta_b200.attention.wan import _top1_branches
    if rank == 0:
        br = _top1_branches(score, 0.3)
        placed = balance.place_units(br, [6.0, 1.6, 1.0], world, balance.max_slots(H, world),
                                     allow_split=balance.split_enabled(world))
        print("mode:", mode, "| exchange:", os.environ.get("VB_ULYSSES", "peer"), "| peer disabled reason:",
              peer.disabled_reason(), "| peer exchanges built:", len(peer._EXCHANGES),
              "| branches:", br, "| units per rank (head, part):", placed, flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
