"""Same workloads through several builds of the library (VB_LIB_PATH is read at import: one subprocess per build).
The builds alternate per round, so each sees the same clocks and power state.  Rates are TFLOP/s, medians of 3 timings.

    python tests/perf_variants.py NAME ...     # vorta_b200/lib/exp/libvb_NAME.so against the in-tree build"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODE = r'''
import os, sys, statistics, torch
sys.path.insert(0, %r)
from vorta_b200 import ops
def timed(fn, iters=10):
    fn(); torch.cuda.synchronize(); ops.timing_enable(True); ops.timing_collect()
    for _ in range(iters): fn()
    torch.cuda.synchronize(); ops.timing_enable(False)
    ms, n, fl = ops.timing_collect(); return ms / iters, fl / iters
W14, W13 = (21, 45, 80), (21, 30, 52)
CASES = (("dense16k", (1, 1, 16384), (1, 1, 16384), (1, 1, 2), 37, [0] * 37),
         ("wan14 full H=8", W14, (3, 9, 16), (3, 3, 2), 8, [0] * 8),
         ("wan14 coreset H=16", W14, (3, 9, 16), (3, 3, 2), 16, [1] * 16),
         ("wan14 sliding H=16", W14, (3, 9, 16), (3, 3, 2), 16, [2] * 16),
         ("wan14mix", W14, (3, 9, 16), (3, 3, 2), 40, [0] * 9 + [1] * 18 + [2] * 13),
         ("wan14 blend H=40", W14, (3, 9, 16), (3, 3, 2), 40, None),
         ("wan14 native sliding (5,9,8) H=16", (20, 45, 80), (5, 9, 8), (2, 3, 2), 16, [2] * 16),
         ("wan13 sliding H=12", W13, (3, 10, 4), (3, 3, 2), 12, [2] * 12),
         ("wan13 mix 4f/4c/4s H=12", W13, (3, 10, 4), (3, 3, 2), 12, [0] * 4 + [1] * 4 + [2] * 4))
out = []
for name, lat, tile, lw, H, branch in CASES:
    plan = ops.Plan(lat, tile, (3, 3, 3) if lat[0] > 1 else (1, 1, 1), lw, 0.5)
    S = plan.seq_len
    q, k, v = (torch.randn((1, S, H, 128), device="cuda").bfloat16().transpose(1, 2) for _ in range(3))
    # branch None: blend mode, every branch on every head weighted by routing scores
    kw = dict(branch=branch) if branch else dict(weights=torch.softmax(torch.randn((1, H, 3), device="cuda"), -1))
    rates = []
    for _ in range(3):
        ms, fl = timed(lambda: ops.routed_attention(plan, q, k, v, **kw))
        rates.append(fl / ms / 1e9)
    out.append("%%s %%.1f" %% (name, statistics.median(rates)))
    del q, k, v, plan
    torch.cuda.empty_cache()
q = torch.randn((1, 75600, 40, 128), device="cuda").bfloat16().transpose(1, 2)
k, v = (torch.randn((1, 512, 40, 128), device="cuda").bfloat16().transpose(1, 2) for _ in range(2))
ms = statistics.median(timed(lambda: ops.attn_dense(q, k, v), iters=20)[0] for _ in range(3))
out.append("wan14 cross attention 40 x 75600 x 512 %%.3f ms" %% ms)
print(" | ".join(out))
''' % ROOT


def main():
    exp = os.path.join(ROOT, "vorta_b200", "lib", "exp")
    builds = [("default (1/8 poly)", None)] + [(n, os.path.join(exp, f"libvb_{n}.so")) for n in sys.argv[1:]]
    for rnd in range(2):
        for name, path in builds:
            env = dict(os.environ)
            if path:
                env["VB_LIB_PATH"] = path
            r = subprocess.run([sys.executable, "-c", CODE], capture_output=True, text=True, env=env, timeout=300)
            print(f"round {rnd} {name:22s} {r.stdout.strip() or r.stderr[-300:]}", flush=True)


if __name__ == "__main__":
    main()
