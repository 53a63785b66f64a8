#!/usr/bin/env python
"""bench.py — DiT denoise-step time of the VORTA-routed Wan 2.1 transformer on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W            # N > 1: launched by torch.distributed.run, one rank per GPU
    python bench.py --impl reference --steps K --warmup W    # the REFERENCE's own processor on the host CPU cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

A "step" is one transformer forward (= one denoise step, no CFG doubling) over one synthetic latent video with
random-init weights of the named architecture.  One JSON line is printed by rank 0 (see README / DESIGN.md section 6
for every field).  Inputs and weights are seeded, so two builds run with the same arguments can be compared output for
output through --dump-outputs.  Workloads (BASELINE.json configs):
    wan14 (default): Wan2.1-T2V-14B, 720p x 81 f -> 21x45x80 = 75,600 tokens, 40 heads, 40 blocks  [configs[2]]
    wan13          : Wan2.1-T2V-1.3B, 480p x 81 f -> 21x30x52 = 32,760 tokens, 12 heads, 30 blocks [configs[1]]
The default is the same for every N so that the driver's 1/2/4/8 scaling ratios compare like with like (12 heads
do not divide by 8); the wan13 numbers are reported next to it at N = 1 in "aux".

CPU legs.  The reference is pure PyTorch; its own files for the path travel to the GPU box under oracle/_ref
(oracle/stage_ref.py).  What a CPU can actually execute in a bench run is BASELINE configs[0]: ONE Wan-1.3B routed
self-attention layer (12 heads, 32,760 tokens) through the reference's WanAttnProcessorTripleEval
(oracle/ref_layer.py).  `--impl reference` executes exactly that, once per step, on every host core — no
extrapolation: its `value` is the measured time of its step, and `cpu_baseline.sample` says what share of the full
workload one such step is.  The GPU arm runs the SAME layer on the same inputs through vorta_b200's processor of the
same name (`like_for_like`, resident and with host buffers) next to the reference timed on the box's cores in the
same run (`cpu_baseline`), and compares the two outputs.  The reference is not part of this repository: where neither
its source (VORTA_REFERENCE_ROOT) nor a staged copy is present, `--impl reference` exits with that message and the GPU
arm reports `cpu_baseline` as unavailable instead of timing anything else under its name.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "wan14": dict(model="wan2.1-t2v-14b", latent=(21, 45, 80), tile=(3, 9, 16), window=(3, 3, 3),
                  lowres_window=(3, 3, 2), rate=0.5, text_tokens=512, heads=40, layers=40,
                  name="Wan2.1-T2V-14B 720p x81f (21x45x80 = 75,600 tokens, 40 heads, 40 blocks), one denoise step"),
    "wan13": dict(model="wan2.1-t2v-1.3b", latent=(21, 30, 52), tile=(3, 10, 4), window=(3, 3, 3),
                  lowres_window=(3, 3, 2), rate=0.5, text_tokens=512, heads=12, layers=30,
                  name="Wan2.1-T2V-1.3B 480p x81f (21x30x52 = 32,760 tokens, 12 heads, 30 blocks), one denoise step"),
}
# contract test only (tests/test_bench_contract.py): tiny grid, 4 heads, 2 blocks; never a reported number
WORKLOADS["tiny"] = dict(model="wan-contract-test", latent=(4, 6, 8), tile=(2, 3, 4), window=(3, 3, 3),
                         lowres_window=(2, 3, 2), rate=0.5, text_tokens=16, heads=4, layers=2,
                         name="CONTRACT TEST ONLY: 2-block 4-head Wan shell, 4x6x8 = 192 tokens")
WORKLOADS["hunyuan"] = dict(model="hunyuanvideo", latent=(33, 45, 80), tile=(3, 9, 16), window=(3, 3, 3),
                            lowres_window=(3, 3, 2), rate=0.5, text_tokens=256, text_valid=64, heads=24, layers=60,
                            name="HunyuanVideo 720p x129f (33x45x80 = 118,800 video tokens + 256 text (64 valid), 24 heads, "
                                 "20 dual + 40 single blocks), one denoise step")
TAU_SPARSE = 0.3          # the reference's inference default (scripts/wan/inference.py:75)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(bf16=float(p.get("bf16_tflops_sustained", p.get("bf16_tflops"))), burst=float(p["bf16_tflops"]),
                    hbm=float(p["hbm_gbs"]), source="MEASURED_PEAKS.json (bf16_tflops_sustained: kernel timed inside a long step)")
    return dict(bf16=1400.0, burst=1590.0, hbm=6650.0, source="fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)")


def recorded_traffic(workload):
    """DRAM bytes (read + write) per launch of the attention kernel for this workload, from the committed
    `ncu --set full` captures (profiles/attn_traffic.json, written by profiles/summarize_full.py --traffic):
    {"self": (bytes, source), "cross": (bytes, source)}; a key is absent when no capture has been committed."""
    path = os.path.join(ROOT, "profiles", "attn_traffic.json")
    out = {}
    try:
        with open(path) as f:
            rec = json.load(f).get(workload) or {}
        for key in ("self", "cross"):
            if key in rec:
                out[key] = (float(rec[key]["dram_bytes_per_launch"]), rec[key]["source"])
    except (OSError, ValueError, KeyError, TypeError):
        pass
    return out


DUMP_BYTES = 64_000_000


def dump_outputs(directory, arrays):
    """Writes each tensor of `arrays` as <directory>/<name>.npy in float32, within DUMP_BYTES in all.  A tensor larger
    than its even share is replaced by a 1-D sample of its flattened elements: one position drawn from a fixed seed in
    each of `share` equal strides, so two runs with the same arguments sample the same positions."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    share = (DUMP_BYTES - 4096 * len(arrays)) // (4 * len(arrays))        # elements; 4 KB left for each .npy header
    for name, t in arrays.items():
        t = t.detach().float().cpu()
        if t.numel() > share:
            edges = torch.arange(share + 1, dtype=torch.float64) * (t.numel() / share)
            u = torch.rand(share, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
            t = t.flatten()[(edges[:-1] + u * (edges[1:] - edges[:-1])).long().clamp_(max=t.numel() - 1)]
        np.save(os.path.join(directory, f"{name}.npy"), t.numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.path = gpu_index, None, f"/tmp/vb_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.out = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "200"], stdout=self.out,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.close()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.remove(self.path)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), power_w_max=max(power), samples=len(sm),
                    reasons=sorted(reasons))


# ------------------------------------------------------------------------------------------------------------
# CPU legs: the REFERENCE's own processor (oracle/_ref or /root/reference) on the host cores, BASELINE configs[0]
# ------------------------------------------------------------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_sample_cfg(wl):
    from oracle import ref_layer as RL
    return RL.TINY if wl is WORKLOADS["tiny"] else RL.CONFIG0


def shared_config(wl, world):
    """`config` of BOTH arms (the reference arm runs "on your arm's config"): the step workload, and the bounded
    sample of it that the CPU legs execute."""
    sample = cpu_sample_cfg(wl)
    return dict(workload=wl["name"], tile=wl["tile"], window=wl["window"], coreset_window=wl["lowres_window"],
                reduction_rate=wl["rate"], tau_sparse=TAU_SPARSE,
                parallelism=f"ulysses{world}" if world > 1 else "single",
                routing="random-init routers, top-1 per head",
                l2="per-step working set (weights + activations) is far larger than the 126 MB L2; no flush needed",
                cpu_sample=f"{sample['name']}; first third of the heads full, second coreset, last sliding tile; coreset "
                           f"window {sample['lowres_window']}, tile {sample['tile']}, window {sample['window']}")


def sample_share(wl):
    """What part of the step workload's routed-attention FLOPs one configs[0] layer is (stated, never applied)."""
    from oracle import ref_layer as RL
    heads, layers = model_dims(wl)
    S = wl["latent"][0] * wl["latent"][1] * wl["latent"][2]
    # uniform 1/3 mix of the BASELINE.md section 3 per-head formulas, for orientation only
    g = wl["lowres_window"][0] * wl["lowres_window"][1] * wl["lowres_window"][2]
    s_c = (S // g) * int(g * (1 - wl["rate"]))
    k_w = 27 * wl["tile"][0] * wl["tile"][1] * wl["tile"][2]
    per_head = 4.0 * 128 * (S * S + s_c * s_c + S * k_w) / 3.0
    return RL.algorithmic_flops(cpu_sample_cfg(wl))["attention"] / (per_head * heads * layers)


def reference_leg(wl, n_timed, n_warm, threads=None, keep_output=False):
    """Run the reference's WanAttnProcessorTripleEval on configs[0]: returns per-call ms list + bookkeeping."""
    from oracle import ref_layer as RL
    cores = threads or host_cores()
    case = RL.build_case(cpu_sample_cfg(wl))
    layer = RL.ReferenceLayer(case, threads=cores)
    prep_s = layer.prepare()
    t0 = time.perf_counter()
    out = None
    for _ in range(max(n_warm, 1)):              # the first call compiles flex_attention for the CPU
        out = layer()
    warm_s = time.perf_counter() - t0
    ms = []
    for _ in range(n_timed):
        t0 = time.perf_counter()
        out = layer()
        ms.append((time.perf_counter() - t0) * 1e3)
    return dict(ms=ms, cores=cores, prepare_s=prep_s, warm_s=warm_s, source=layer.source, case=case,
                out=out if keep_output else None, flops=RL.algorithmic_flops(cpu_sample_cfg(wl)))


def reference_missing():
    """None when the reference's own files can be imported, else why not (the reference is not part of this
    repository, and nothing else is timed under its name)."""
    from oracle import ref_loader
    if ref_loader.available():
        return None
    return ("reference not available: neither VORTA_REFERENCE_ROOT (a checkout of wenhao728/VORTA) nor a staged copy "
            "under oracle/_ref (oracle/stage_ref.py)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                   # rank 0 alone runs the CPU arm; the other ranks exit 0
    missing = reference_missing()
    if missing:
        raise SystemExit(f"bench.py --impl reference: {missing}")
    cores = host_cores()
    os.environ["OMP_NUM_THREADS"] = str(cores)   # torchrun exports OMP_NUM_THREADS=1; must be set before torch loads
    os.environ["MKL_NUM_THREADS"] = str(cores)
    wl = WORKLOADS[args.workload]
    r = reference_leg(wl, args.steps, args.warmup, threads=cores, keep_output=bool(args.dump_outputs))
    value = statistics.mean(r["ms"])
    share = sample_share(wl)
    sample = (f"each step = ONE real call of the reference's own WanAttnProcessorTripleEval "
              f"(vorta/attention/wan.py:303-438, files from {'oracle/_ref' if r['source'] == 'staged' else '/root/reference'}) "
              f"on BASELINE configs[0] (fp32 up-cast of the bf16 inputs, {cores} threads): "
              f"{r['flops']['total'] / 1e12:.2f} TFLOP algorithmic = about 1/{1.0 / share:.0f} of the routed attention "
              f"of one step of the workload; value is the measured time of that step, NOT scaled to the workload; "
              f"untimed: block-mask build {r['prepare_s']:.0f} s + {max(args.warmup, 1)} warm-up calls {r['warm_s']:.0f} s")
    line = dict(impl="reference", metric="dit_denoise_step_ms", value=value, unit="ms", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=value, higher_is_better=False, scaling="strong",
                vs_baseline=None, dtype="f32", data="synthetic (storage-free hashed bf16-exact values)",
                config=shared_config(wl, args.gpus),
                cpu_baseline=dict(value=value, unit="ms", cores=cores, kind="reference", sample=sample,
                                  ms_min=min(r["ms"]), ms_max=max(r["ms"]),
                                  tflops=r["flops"]["total"] / (value * 1e-3) / 1e12),
                like_for_like=dict(workload="BASELINE configs[0]", reference_cpu_ms=value),
                e2e=dict(value=value, unit="ms", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(hidden_states=r["out"]))
    print(json.dumps(line), flush=True)


def branch_counts(branches):
    c = [0, 0, 0]
    for layer in branches:
        for e in layer:
            c[e] += 1
    return c


def model_dims(wl):
    """(heads, attention layers) of the workload's architecture (the reference arm must not import vorta_b200)."""
    return wl["heads"], wl["layers"]


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def build_model(wl, device):
    import torch
    if wl["model"] == "hunyuanvideo":
        from vorta_b200.dit import HunyuanDiT
        from vorta_b200.patch import modeling_hunyuan, prepare_hunyuan_self_attn_kwargs
        model = HunyuanDiT.build(wl["model"], device, torch.bfloat16, seed=0)
        modeling_hunyuan.apply_vorta_transformer(model, train_router=False, router_dtype=torch.float32)
        kw = prepare_hunyuan_self_attn_kwargs(
            dict(latent_shape=wl["latent"], window_size=wl["window"], tile_size=wl["tile"],
                 lowres_window_size=wl["lowres_window"], lowres_reduction_rate=wl["rate"]), device, tau_sparse=TAU_SPARSE)
        return model, kw
    from vorta_b200.dit import WanDiT
    from vorta_b200.patch import apply_vorta_transformer, prepare_wan_self_attn_kwargs
    model = WanDiT.build(wl["model"], device, torch.bfloat16, seed=0)
    apply_vorta_transformer(model, train_router=False, router_dtype=torch.float32)
    kw = prepare_wan_self_attn_kwargs(
        dict(latent_shape=wl["latent"], window_size=wl["window"], tile_size=wl["tile"],
             lowres_window_size=wl["lowres_window"], lowres_reduction_rate=wl["rate"]), device, tau_sparse=TAU_SPARSE)
    return model, kw


def host_inputs(wl, cfg):
    import torch
    g = torch.Generator().manual_seed(1234)
    T, H, W = wl["latent"]
    lat = torch.randn((1, cfg.in_channels, T, 2 * H, 2 * W), generator=g).to(torch.bfloat16).pin_memory()
    text_dim = cfg.text_embed_dim if hasattr(cfg, "text_embed_dim") else cfg.text_dim
    txt = torch.randn((1, wl["text_tokens"], text_dim), generator=g).to(torch.bfloat16).pin_memory()
    ts = torch.tensor([500.0]).pin_memory()
    return lat, txt, ts


def make_step(model, wl, device, kw):
    """Returns call(latents, timestep, text) -> model outputs for the workload's model family."""
    import torch
    if wl["model"] != "hunyuanvideo":
        return lambda lat, ts, txt, **extra: model(lat, ts, txt, self_attention_kwargs=kw, return_dict=False, **extra)
    g = torch.Generator().manual_seed(99)
    mask = torch.zeros((1, wl["text_tokens"]), dtype=torch.bool, device=device)
    mask[:, :wl["text_valid"]] = True
    pooled = torch.randn((1, model.config.pooled_projection_dim), generator=g).to(device, torch.bfloat16)
    guidance = torch.tensor([6000.0], device=device)
    return lambda lat, ts, txt, **extra: model(lat, ts, txt, mask, pooled, guidance, self_attention_kwargs=dict(kw),
                                               return_dict=False, **extra)


def time_steps(fn, steps, warmup, dist_on, profile=False, after_warmup=None):
    import torch
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    if after_warmup is not None:
        after_warmup()
    if profile:          # ncu --profile-from-start off: capture exactly one warmed-up step, outside the timing
        torch.cuda.cudart().cudaProfilerStart()
        fn()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        if after_warmup is not None:
            after_warmup()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    ms = e0.elapsed_time(e1) / steps
    if dist_on:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def run_workload(wl, args, rank, world, device, with_e2e=True):
    import torch
    import torch.distributed as dist
    from vorta_b200 import ops
    dist_on = world > 1
    model, kw = build_model(wl, device)
    cfg = model.config
    lat_h, txt_h, ts_h = host_inputs(wl, cfg)
    lat_d, txt_d, ts_d = lat_h.to(device), txt_h.to(device), ts_h.to(device)
    out_h = torch.empty(lat_h.shape, dtype=torch.bfloat16).pin_memory()

    call = make_step(model, wl, device, kw)

    last = {}

    @torch.no_grad()
    def step_resident():
        out = call(lat_d, ts_d, txt_d)[0]
        if args.dump_outputs:          # kept only for a dump: holding it across steps changes what the allocator reuses
            last["sample"] = out
        return out

    @torch.no_grad()
    def step_e2e():
        a = lat_h.to(device, non_blocking=True)
        b = txt_h.to(device, non_blocking=True)
        c = ts_h.to(device, non_blocking=True)
        out = call(a, c, b)[0]
        out_h.copy_(out, non_blocking=True)
        return out

    # routing mix of this run (one untimed forward): the fp32 top-1 decisions the kernels actually ran with.  (The
    # reference-shaped `routing_scores` output is rounded to the activation dtype; with random-init routers every score
    # is ~1/3 and bf16 ties flip the argmax of ~5 % of the heads: round 1 counted 552 / 568 / 480 where the kernels ran
    # a different mix, which is the 2181 vs 2279 TFLOP / step discrepancy of VERDICT.md.)
    with torch.no_grad():
        call(lat_d, ts_d, txt_d)
    counts = branch_counts(model._vb_last_branches)

    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    ops.timing_enable(True)

    def reset_counters():          # the timers and launch counters cover EXACTLY the timed steps
        ops.timing_collect()
        ops.stats_reset()
        if dist_on:
            from vorta_b200.ulysses import peer
            peer.nvlink_tx_bytes(reset=True)

    sampler.start()
    ms = time_steps(step_resident, args.steps, args.warmup, dist_on, profile=args.profile, after_warmup=reset_counters)
    clocks = sampler.stop()
    outputs = {name: t.float().cpu() for name, t in last.items()} if args.dump_outputs else None
    ops.timing_enable(False)
    kinds = ops.timing_collect_kinds()
    launches_step = ops.stats()[0] / args.steps
    nvlink_tx_step = None
    if dist_on:
        from vorta_b200.ulysses import peer
        nvlink_tx_step = peer.nvlink_tx_bytes() / args.steps
    per = {}
    for name, (k_ms, k_n, k_fl) in kinds.items():
        per[name] = dict(ms_step=k_ms / args.steps, launches_step=k_n / args.steps, flops_step=k_fl / args.steps)
    attn_ms_step = sum(v["ms_step"] for v in per.values())
    attn_flops_step = sum(v["flops_step"] for v in per.values())
    e2e_ms = time_steps(step_e2e, args.steps, 1, dist_on) if with_e2e else None
    # whole-job attention flops: ranks hold disjoint head chunks
    if dist_on:
        t = torch.tensor([attn_flops_step, attn_ms_step], device="cuda", dtype=torch.float64)
        fl = t.clone(); dist.all_reduce(fl, op=dist.ReduceOp.SUM)
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        job_flops, attn_ms_max = float(fl[0].item()), float(mx[1].item())
        each = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(each, t)
        attn_ms_ranks = [round(float(e[1].item()), 3) for e in each]
    else:
        job_flops, attn_ms_max = attn_flops_step, attn_ms_step
        attn_ms_ranks = None
    # closed-form cross-check of the library's FLOP counter: head counts x BASELINE.md section 3 formulas (+ the dense
    # cross-attention launches of the Wan blocks: 4 * S * text * 128 per head)
    heads, layers = model_dims(wl)
    S = wl["latent"][0] * wl["latent"][1] * wl["latent"][2]
    plan_kw = dict(text_len=wl["text_tokens"], text_valid=wl.get("text_valid", 0)) if wl["model"] == "hunyuanvideo" else {}
    plan = ops.Plan(wl["latent"], wl["tile"], wl["window"], wl["lowres_window"], wl["rate"], **plan_kw)
    formula = sum(counts[e] * plan.flops_per_head(e) for e in range(3))
    if wl["model"] != "hunyuanvideo":
        formula += 4.0 * S * wl["text_tokens"] * 128 * heads * layers
    del model
    torch.cuda.empty_cache()
    return dict(ms=ms, e2e_ms=e2e_ms, clocks=clocks, counts=counts, attn_ms_step=attn_ms_step,
                attn_flops_step=attn_flops_step, per_kind=per, launches_step=launches_step, job_flops=job_flops,
                attn_ms_max=attn_ms_max, attn_ms_ranks=attn_ms_ranks, nvlink_tx_step=nvlink_tx_step,
                formula_flops_step=formula, outputs=outputs,
                h2d=lat_h.numel() * 2 + txt_h.numel() * 2 + 4, d2h=out_h.numel() * 2, cfg=cfg)


# ------------------------------------------------------------------------------------------------------------
# like-for-like leg (N = 1): BASELINE configs[0] on the GPU through the reference-facing processor, next to the
# reference's own processor on the host cores in the same run
# ------------------------------------------------------------------------------------------------------------
def like_for_like_leg(args, device, with_cpu=True):
    import torch
    from oracle import ref_layer as RL                  # input generator + the CPU checker / baseline of this leg
    from vorta_b200.attention import WanAttnProcessorTripleEval, get_group_info
    cfg = cpu_sample_cfg(WORKLOADS[args.workload])
    case = RL.build_case(cfg)
    attn = case["attn"].to(device, torch.bfloat16)
    hs_h = case["hidden_states"].to(torch.bfloat16).pin_memory()
    score_h = case["routing_score"].pin_memory()
    rot = case["rotary_emb"].to(device)
    hs_d = hs_h.to(device)
    score_d = score_h.to(device)
    out_h = torch.empty(hs_h.shape, dtype=torch.bfloat16).pin_memory()
    proc = WanAttnProcessorTripleEval(check_input=True)
    kw = dict(lowres_group_info=get_group_info(cfg["latent"], cfg["lowres_window"], cfg["rate"], device=device),
              flex_attn_mask_func=None, window_size=cfg["window"], tile_size=cfg["tile"], latent_shape=cfg["latent"])

    def resident():
        return proc(attn, hs_d, None, None, rot, tau_sparse=cfg["tau_sparse"], routing_score=score_d, **kw)

    def e2e():
        a = hs_h.to(device, non_blocking=True)
        b = score_h.to(device, non_blocking=True)
        out = proc(attn, a, None, None, rot, tau_sparse=cfg["tau_sparse"], routing_score=b, **kw)
        out_h.copy_(out, non_blocking=True)
        return out

    n = max(args.steps, 10)
    ms = time_steps(resident, n, 3, False)
    e2e_ms = time_steps(e2e, n, 3, False)
    flops = RL.algorithmic_flops(cfg)
    res = dict(workload=cfg["name"], gpu_ms=ms, gpu_e2e_ms=e2e_ms, calls=n,
               h2d_bytes_per_call=hs_h.numel() * 2 + score_h.numel() * 4, d2h_bytes_per_call=out_h.numel() * 2,
               gpu_tflops=flops["total"] / (ms * 1e-3) / 1e12,
               api="vorta_b200.attention.WanAttnProcessorTripleEval.__call__ (the reference's processor signature)")
    cpu = None
    missing = reference_missing() if with_cpu else None
    if missing:
        cpu = dict(kind="reference", available=False, value=None, unit="ms", reason=missing)
    elif with_cpu:
        out_gpu = resident().float().cpu()
        r = reference_leg(WORKLOADS[args.workload], 2, 1, keep_output=True)
        ref = r["out"].float()
        a64, b64 = out_gpu.flatten().double(), ref.flatten().double()
        cos = float((a64 @ b64) / (a64.norm() * b64.norm()))
        err = (out_gpu - ref).abs().max().item()
        cpu_ms = statistics.mean(r["ms"])
        cpu = dict(value=cpu_ms, unit="ms", cores=r["cores"], kind="reference",
                   sample=(f"the reference's own WanAttnProcessorTripleEval (vorta/attention/wan.py:303-438, files from "
                           f"{'oracle/_ref' if r['source'] == 'staged' else '/root/reference'}) on BASELINE configs[0], fp32 up-cast of "
                           f"the same bf16 inputs as like_for_like.gpu_ms, {r['cores']} threads, mean of 2 timed calls "
                           f"after 1 warm-up; NOT scaled to the step workload (one such layer is about "
                           f"1/{1.0 / sample_share(WORKLOADS[args.workload]):.0f} of its routed attention); untimed: block-mask "
                           f"build {r['prepare_s']:.0f} s, warm-up {r['warm_s']:.0f} s"),
                   ms_calls=r["ms"], tflops=flops["total"] / (cpu_ms * 1e-3) / 1e12)
        res.update(reference_cpu_ms=cpu_ms, speedup_resident=cpu_ms / ms, speedup_e2e=cpu_ms / e2e_ms,
                   parity=dict(cosine=cos, max_abs=err, ref_abs_max=ref.abs().max().item(),
                               note="bf16 GPU layer (bf16 projections, RMSNorm, RoPE, attention) vs the fp32 reference "
                                    "layer on identical inputs"))
    return res, cpu


def ulysses_parity_hunyuan(wl, device, world, rank):
    """HunyuanVideo: the joint [video | text] attention of one layer (video tokens sharded, text replicated; K / V
    pooled with K's own matching) through the sequence-parallel path vs rank 0's single-GPU call, bit for bit
    (reference semantics: vorta/attention/hunyuan.py:136-189 around :410-507)."""
    import torch
    import torch.distributed as dist
    from vorta_b200 import _lib as L
    from vorta_b200 import ops
    from vorta_b200.attention.hunyuan import HunyuanVideoFlashAttnProcessorTripleEval
    from vorta_b200.ulysses import SP_STATE, all_gather, peer
    heads, _ = model_dims(wl)
    TL, TV = wl["text_tokens"], wl["text_valid"]
    plan = ops.Plan(wl["latent"], wl["tile"], wl["window"], wl["lowres_window"], wl["rate"], text_len=TL, text_valid=TV)
    S = plan.seq_len
    s_loc = S // world
    g = torch.Generator().manual_seed(4321)
    branch = [(h * 7 + 1) % 3 for h in range(heads)]
    q, k, v = (torch.randn((1, S + TL, heads, 128), generator=g).to(torch.bfloat16).to(device).transpose(1, 2)
               for _ in range(3))
    proc = HunyuanVideoFlashAttnProcessorTripleEval()

    def shard(t):          # this rank's video tokens followed by the replicated text tokens
        return torch.cat([t[:, :, rank * s_loc:(rank + 1) * s_loc], t[:, :, S:]], dim=2)

    video, text = proc._joint_attention(shard(q), shard(k), shard(v), plan, TL, branch=branch,
                                        flags=L.ATTN_CORESET_KV_FROM_K)
    got = torch.cat([all_gather(video.transpose(1, 2).contiguous(), dim=1), text.transpose(1, 2)], dim=1)
    res = None
    if rank == 0:
        en, sz = SP_STATE._enabled, SP_STATE._sp_size
        SP_STATE._enabled, SP_STATE._sp_size = False, 1
        try:
            ref = ops.routed_attention(plan, q, k, v, branch=branch, flags=L.ATTN_CORESET_KV_FROM_K).transpose(1, 2)
        finally:
            SP_STATE._enabled, SP_STATE._sp_size = en, sz
        err = (got.float() - ref.float()).abs().max().item()
        res = dict(equal=bool(torch.equal(got, ref)), max_abs=err,
                   what=f"one routed joint-attention layer, {heads} heads x ({S} video + {TL} text, {TV} valid) tokens, "
                        f"branches (7h+1)%3, {world}-rank Ulysses path vs rank 0's single-GPU call on the same q, k, v",
                   exchange="nvlink-peer" if (os.environ.get("VB_ULYSSES", "peer") != "nccl"
                                             and peer.disabled_reason() is None) else "nccl")
    torch.cuda.synchronize()
    dist.barrier()
    del q, k, v, got, video, text
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------------------
# N > 1: the Ulysses path that is about to be timed == the single-GPU call, at the workload's real size
# ------------------------------------------------------------------------------------------------------------
def ulysses_parity(wl, device, world, rank):
    """One routed self-attention layer at the workload's full geometry and head count: every rank holds the same
    seeded q, k, v; the sequence-parallel path (token shards in, NVLink peer / NCCL exchange, this rank's heads,
    exchange out, all-gather of the token shards) must reproduce rank 0's single-GPU vb_attn_fwd BIT FOR BIT
    (reference semantics: vorta/ulysses/utils.py:15-124 around wan.py:243-294)."""
    import torch
    import torch.distributed as dist
    from vorta_b200 import ops
    from vorta_b200.attention.wan import WanAttnProcessorTripleEval
    from vorta_b200.ulysses import SP_STATE, all_gather, peer
    if wl["model"] == "hunyuanvideo":
        return ulysses_parity_hunyuan(wl, device, world, rank)
    heads, _ = model_dims(wl)
    plan = ops.Plan(wl["latent"], wl["tile"], wl["window"], wl["lowres_window"], wl["rate"])
    S = plan.seq_len
    s_loc = S // world
    g = torch.Generator().manual_seed(4321)
    branch = [(h * 7 + 1) % 3 for h in range(heads)]
    q, k, v = (torch.randn((1, S, heads, 128), generator=g).to(torch.bfloat16).to(device).transpose(1, 2)
               for _ in range(3))
    proc = WanAttnProcessorTripleEval()
    sl = slice(rank * s_loc, (rank + 1) * s_loc)
    mine = proc._routed_attention(q[:, :, sl], k[:, :, sl], v[:, :, sl], plan, branch=branch)   # (1, H, S_loc, 128)
    got = all_gather(mine.transpose(1, 2).contiguous(), dim=1)                                    # (1, S, H, 128)
    res = None
    if rank == 0:
        en, sz = SP_STATE._enabled, SP_STATE._sp_size
        SP_STATE._enabled, SP_STATE._sp_size = False, 1
        try:
            ref = ops.routed_attention(plan, q, k, v, branch=branch).transpose(1, 2)
        finally:
            SP_STATE._enabled, SP_STATE._sp_size = en, sz
        err = (got.float() - ref.float()).abs().max().item()
        res = dict(equal=bool(torch.equal(got, ref)), max_abs=err,
                   what=f"one routed self-attention layer, {heads} heads x {S} tokens, branches (7h+1)%3, "
                        f"{world}-rank Ulysses path vs rank 0's single-GPU call on the same q, k, v",
                   exchange="nvlink-peer" if (os.environ.get("VB_ULYSSES", "peer") != "nccl"
                                             and peer.disabled_reason() is None) else "nccl")
    torch.cuda.synchronize()
    dist.barrier()
    del q, k, v, got, mine
    torch.cuda.empty_cache()
    return res


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from vorta_b200 import _lib as L
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: vorta_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    L.check(L.lib().vb_device_check())
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
        from vorta_b200.ulysses import SP_STATE
        SP_STATE.setup_sp_group(world)
    wl = WORKLOADS[args.workload]
    parity = ulysses_parity(wl, device, world, rank) if world > 1 else None
    r = run_workload(wl, args, rank, world, device)
    peaks = measured_peaks()

    def rate(flops, ms):
        return flops / (ms * 1e-3) / 1e12 if ms > 0 else 0.0

    routed, dense = r["per_kind"]["routed"], r["per_kind"]["dense"]
    achieved = rate(routed["flops_step"], routed["ms_step"])       # the dominant kernel launch: a layer's routed self-attention
    achieved_all = rate(r["attn_flops_step"], r["attn_ms_step"])
    traffic = recorded_traffic(args.workload)
    config = shared_config(wl, world)
    line = dict(
        metric="dit_denoise_step_ms", value=r["ms"], unit="ms", n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=r["ms"], higher_is_better=False, scaling="strong", vs_baseline=None, dtype="bf16",
        data="synthetic (seeded N(0,1) latents / text embeddings, random-init weights)",
        config=config,
        routing_mix=dict(heads_per_branch_all_layers=dict(full=r["counts"][0], coreset=r["counts"][1],
                                                          sliding=r["counts"][2])),
        routed_attn_effective_tflops=rate(r["job_flops"], r["attn_ms_max"]),
        attn_kernel_ms_per_step=r["attn_ms_step"],
        attn_flops_per_step=dict(library_counter=r["attn_flops_step"], closed_form=r["formula_flops_step"],
                                 routed_launches=routed["flops_step"], dense_launches=dense["flops_step"],
                                 note="library counter = sum over the timed launches of this rank; closed form = head counts x "
                                      "BASELINE.md section 3 formulas (+ 4*S*512*128 per head per block of dense cross attention)"
                                      + (", whole job" if world > 1 else "")),
        roofline=dict(bound="tensor", achieved=achieved, peak=peaks["bf16"], unit="TFLOP/s",
                      frac=achieved / peaks["bf16"], traffic=traffic.get("self", (None, None))[0],
                      traffic_unit="bytes / launch (DRAM read + write)", traffic_source=traffic.get("self", (None, None))[1],
                      kernel="vb_attn_fwd_kernel (routed self-attention launch: a layer's full + coreset + sliding heads in one grid)",
                      ms_per_launch=routed["ms_step"] / max(routed["launches_step"], 1),
                      launches_per_step=routed["launches_step"], ms_per_step=routed["ms_step"],
                      frac_of_burst=achieved / peaks["burst"], frac_of_spec_2250=achieved / 2250.0,
                      peak_source=peaks["source"],
                      cross_attention=dict(
                          kernel="vb_attn_fwd_kernel (dense launch: 512 text keys per query)",
                          achieved=rate(dense["flops_step"], dense["ms_step"]), unit="TFLOP/s",
                          ms_per_launch=dense["ms_step"] / max(dense["launches_step"], 1),
                          launches_per_step=dense["launches_step"], ms_per_step=dense["ms_step"],
                          traffic=traffic.get("cross", (None, None))[0],
                          hbm_gbs=(traffic["cross"][0] / (dense["ms_step"] / max(dense["launches_step"], 1) * 1e-3) / 1e9
                                   if traffic.get("cross", (None, None))[0] and dense["ms_step"] > 0 else None),
                          hbm_peak_gbs=peaks["hbm"]),
                      all_attention_launches=dict(achieved=achieved_all, frac=achieved_all / peaks["bf16"])),
        clocks=r["clocks"],
        e2e=dict(value=r["e2e_ms"], unit="ms", h2d_bytes_per_step=r["h2d"], d2h_bytes_per_step=r["d2h"]),
        gpu_launches=int(round(r["launches_step"] * args.steps)),
    )
    if parity is not None:
        line["parity"] = parity
    if r["attn_ms_ranks"] is not None:        # attention kernel time per rank: the placement's balance, measured
        line["attn_kernel_ms_per_rank"] = r["attn_ms_ranks"]
        line["nvlink"] = dict(
            tx_bytes_per_step_rank0=r["nvlink_tx_step"], tx_gbs_rank0=r["nvlink_tx_step"] / (r["ms"] * 1e-3) / 1e9,
            note="bytes rank 0 stores into peers' exchange buffers per step (Q/K/V rows in, output rows out), counted from "
                 "the placement tables: `nvidia-smi nvlink -gt d` reads N/A on this pool; average rate over the whole step, "
                 "peak NVLink 5 = 900 GB/s per direction")
    if world == 1 and rank == 0:
        if not args.no_cpu_baseline:
            lfl, cpu = like_for_like_leg(args, device, with_cpu=True)
            line["like_for_like"] = lfl
            line["cpu_baseline"] = cpu
        if args.workload == "wan14" and not args.no_aux:
            a = run_workload(WORKLOADS["wan13"], args, rank, world, device, with_e2e=True)
            ar = a["per_kind"]["routed"]
            ach = rate(ar["flops_step"], ar["ms_step"])
            line["aux"] = dict(workload=WORKLOADS["wan13"]["name"], ms_per_step=a["ms"], e2e_ms=a["e2e_ms"],
                               heads_per_branch_all_layers=dict(full=a["counts"][0], coreset=a["counts"][1],
                                                                sliding=a["counts"][2]),
                               attn_kernel_ms_per_step=a["attn_ms_step"], routed_attn_tflops=ach,
                               roofline_frac=ach / peaks["bf16"],
                               cross_attn_tflops=rate(a["per_kind"]["dense"]["flops_step"],
                                                      a["per_kind"]["dense"]["ms_step"]))
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, r["outputs"])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vorta_b200", choices=["vorta_b200", "reference"])
    ap.add_argument("--workload", default="wan14", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true")
    ap.add_argument("--profile", action="store_true", help="bracket one warmed-up step with cudaProfilerStart/Stop")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
