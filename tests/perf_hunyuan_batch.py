"""Cost of batching HunyuanVideo prompts of different lengths: one 720p x 129-frame routed layer (latent 33 x 45 x 80,
24 heads, text_len 256) at batch 2 with text lengths (64, 200), against two batch-1 calls with those lengths.
CUDA events around each variant, alternated, warm-up first.  Prints one JSON line with the card and its power limit.

Usage: python tests/perf_hunyuan_batch.py [--iters N]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vorta_b200 import _lib as L  # noqa: E402
from vorta_b200 import ops  # noqa: E402

LAT, TILE, WIN, LW, TL, H = (33, 45, 80), (3, 9, 16), (3, 3, 3), (3, 3, 2), 256, 24
LENGTHS = (64, 200)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    L.check(L.lib().vb_device_check())
    dev = torch.device("cuda:0")
    S = LAT[0] * LAT[1] * LAT[2]
    g = torch.Generator().manual_seed(0)
    q, k, v = (torch.randn((2, S + TL, H, 128), generator=g).to(dev, torch.bfloat16).transpose(1, 2) for _ in range(3))
    # a routed mix like a mid-denoise layer: 6 full, 8 coreset, 10 sliding heads
    branch = [0] * 6 + [1] * 8 + [2] * 10
    branch = [branch[(h * 7) % H] for h in range(H)]
    plans = {tv: ops.Plan(LAT, TILE, WIN, LW, 0.5, text_len=TL, text_valid=tv) for tv in LENGTHS}
    out2 = torch.empty((2, S + TL, H, 128), dtype=torch.bfloat16, device=dev).transpose(1, 2)
    flags = L.ATTN_CORESET_KV_FROM_K

    def batched():
        ops.routed_attention(plans[LENGTHS[0]], q, k, v, branch=branch, flags=flags, out=out2, text_valid=list(LENGTHS))

    def separate():
        for b, tv in enumerate(LENGTHS):
            ops.routed_attention(plans[tv], q[b:b + 1], k[b:b + 1], v[b:b + 1], branch=branch, flags=flags,
                                 out=out2[b:b + 1])

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    for _ in range(2):
        batched()
        separate()
    torch.cuda.synchronize()
    ref = out2.clone()
    batched()
    torch.cuda.synchronize()
    equal = torch.equal(ref, out2)
    t_b, t_s = [], []
    for _ in range(args.iters):
        t_b.append(timed(batched))
        t_s.append(timed(separate))
    t_b.sort()
    t_s.sort()
    res = dict(card=card(), layer="hunyuan 720p x 129f routed, 24 heads (6 full / 8 coreset / 10 sliding)",
               lengths=list(LENGTHS), batch2_ms_median=t_b[len(t_b) // 2], two_batch1_ms_median=t_s[len(t_s) // 2],
               batch2_ms_min=t_b[0], two_batch1_ms_min=t_s[0], ratio=t_b[len(t_b) // 2] / t_s[len(t_s) // 2],
               outputs_equal=equal, iters=args.iters)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
