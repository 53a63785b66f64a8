"""Multi-GPU check of HunyuanVideo at batch 2 with per-sample text lengths, launched by torchrun (one rank per GPU).

The same Q / K / V go through the Ulysses NCCL path (batch > 1 always takes it) and through one single-GPU call; the
gathered outputs must be bit-identical, for top-1 (Eval), blend (Train) and dense (use_original_attn) attention.
Prints one line per case; exits non-zero on a mismatch.  Driven by tests/test_multigpu_hunyuan_batch.py."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vorta_b200 import _lib as L  # noqa: E402
from vorta_b200 import ops  # noqa: E402
from vorta_b200.attention import HunyuanVideoFlashAttnProcessorTripleEval  # noqa: E402
from vorta_b200.attention._plans import get_plan  # noqa: E402
from vorta_b200.ulysses import SP_STATE, all_gather  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ok = True

    lat, tile, win, lw, TL = (4, 8, 8), (2, 4, 4), (3, 3, 3), (2, 2, 2), 40
    S, H, tvs = lat[0] * lat[1] * lat[2], 4 * world, [29, 6]
    g = torch.Generator().manual_seed(3)
    q, k, v = (torch.randn((2, S + TL, H, 128), generator=g).to(dev, torch.bfloat16).transpose(1, 2) for _ in range(3))
    weights = torch.softmax(torch.randn((2, H, 3), generator=g) * 2, -1).to(dev)
    branch = [(h * 7 + 1) % 3 for h in range(H)]
    plan = get_plan(lat, tile, win, lw, int(8 * 0.5) - 1, TL, tvs[0])
    dense = get_plan((1, 1, S), (1, 1, S), (1, 1, 1), (1, 1, 1), 0, TL, tvs[0])
    cases = [("top-1 (eval)", plan, dict(branch=branch, flags=L.ATTN_CORESET_KV_FROM_K)),
             ("blend (train)", plan, dict(weights=weights, flags=L.ATTN_CORESET_KV_FROM_K)),
             ("dense (use_original_attn)", dense, dict(branch=[L.BRANCH_FULL] * H))]
    proc = HunyuanVideoFlashAttnProcessorTripleEval()
    s_loc = S // world

    def shard(t):          # this rank's video tokens followed by the replicated text tokens
        return torch.cat([t[:, :, rank * s_loc:(rank + 1) * s_loc], t[:, :, S:]], dim=2)

    with torch.no_grad():
        refs = [ops.routed_attention(p, q, k, v, text_valid=tvs, **kw) for _, p, kw in cases]
        SP_STATE.setup_sp_group(world)
        for (name, p, kw), ref in zip(cases, refs):
            video, text = proc._joint_attention(shard(q), shard(k), shard(v), p, TL, text_valid=tvs, **kw)
            got = torch.cat([all_gather(video.transpose(1, 2).contiguous(), dim=1), text.transpose(1, 2)], dim=1)
            good = torch.equal(got, ref.transpose(1, 2))
            ok &= good
            if rank == 0:
                print(f"hunyuan batch 2, text_valid {tvs}, {name:28s} world {world}: "
                      f"{'OK (bit-identical)' if good else 'MISMATCH'}", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
