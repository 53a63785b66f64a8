"""Coreset selection at the Wan-14B grid (latent 21 x 45 x 80, 40 heads): the shared-memory kernel for large groups
(g = 48 as (3, 1, 16), g = 60 as (3, 5, 4); 64-token windows do not divide 21 x 45 x 80, so g = 64 runs as (4, 1, 16)
on the reference's own 20 x 45 x 80 grid) beside the warp kernel at the production window (3, 3, 2), in one process
on one card.  Inputs are N(0, 1) and spatially smooth (cosines 0.99+, more groups take the fp64 recheck) activations
in the (B, S, H, 128) memory the projections produce; 40 heads x S x 256 B = 774 MB per pass, beyond the 126 MB L2.
CUDA events around `iters` calls, the variants alternated per round, warm-up first; median of the rounds.
HBM bytes counted per call: every token row read once (S x 256 B per head) + the four int tables written.
Prints one JSON line per case with the card and its power limit; no threshold.

Usage: python tests/perf_select_large.py [--iters N] [--rounds R]"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vorta_b200 import _lib as L  # noqa: E402
from vorta_b200 import ops  # noqa: E402

from perf_hunyuan_batch import card  # noqa: E402

H = 40
CASES = [   # name, latent, lowres window
    ("warp kernel (3,3,2) g=18", (21, 45, 80), (3, 3, 2)),
    ("smem kernel (3,1,16) g=48", (21, 45, 80), (3, 1, 16)),
    ("smem kernel (3,5,4) g=60", (21, 45, 80), (3, 5, 4)),
    ("smem kernel (4,1,16) g=64 @20x45x80", (20, 45, 80), (4, 1, 16)),
]


def table_bytes(plan):
    G, n_u, n_p = plan.num_groups, plan.n_unpooled, plan.num_pooled
    return H * (plan.seq_len * 256 + G * (n_u + n_p) * 8 + plan.coreset_len * 4 + G * n_p * 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    L.check(L.lib().vb_device_check())
    dev = torch.device("cuda:0")
    inputs = {}
    for name, lat, lw in CASES:
        plan = ops.Plan(lat, (1, 1, 1), (1, 1, 1), lw, 0.5)
        S = plan.seq_len
        g = torch.Generator(device=dev).manual_seed(S)
        x = torch.randn((1, S, H, 128), generator=g, device=dev)
        smooth = torch.randn((1, 1, H, 128), generator=g, device=dev) + 0.05 * x
        inputs[name] = (plan, {"randn": x.to(torch.bfloat16).transpose(1, 2),
                               "smooth": smooth.to(torch.bfloat16).transpose(1, 2)})
    times = {(n, kind): [] for n in inputs for kind in ("randn", "smooth")}
    for key in times:                                      # warm-up
        plan, xs = inputs[key[0]]
        ops.coreset_select(plan, xs[key[1]], want_tokens=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    for _ in range(args.rounds):
        for key in times:
            plan, xs = inputs[key[0]]
            x = xs[key[1]]
            e0.record()
            for _ in range(args.iters):
                ops.coreset_select(plan, x, want_tokens=True)
            e1.record()
            torch.cuda.synchronize()
            times[key].append(e0.elapsed_time(e1) / args.iters)
    where = card()
    for (name, kind), ts in times.items():
        plan = inputs[name][0]
        ms = statistics.median(ts)
        nbytes = table_bytes(plan)
        print(json.dumps({"case": name, "input": kind, "latent": list(plan_lat(name)), "heads": H,
                          "group_size": plan.group_size, "ms": round(ms, 4), "ms_min": round(min(ts), 4),
                          "ms_max": round(max(ts), 4), "bytes": nbytes, "TB_per_s": round(nbytes / ms / 1e9, 3),
                          "card": where}))


def plan_lat(name):
    return next(lat for n, lat, _ in CASES if n == name)


if __name__ == "__main__":
    main()
