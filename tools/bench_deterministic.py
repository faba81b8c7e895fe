"""What deterministic mode costs on the GPU, in one process (the card's name and power limit are read in the same run):

  * the graphed training step (full 331-pathway model, eval) at 10k and 32k tiles, default against deterministic,
    replays alternated A / B after a warm-up;
  * one call of mt_dilated_attn_bwd, impl 2 (the default persistent backward) against impl 4 (deterministic), at the
    same sizes, alternated;
  * the kernels of impl 4 (torch.profiler, CUDA activities): the dQ kernel's algorithmic FLOP/s (S + dP + dQ = 1.5 x the
    forward's FLOPs) and its share of the dense bf16 peak of the data sheet (2 250 TFLOP/s for one B200 at 1 000 W).

    python tools/bench_deterministic.py [--steps 20] [--out DIR]

Every time is the median of CUDA-event timings with the min / max beside it.  Inputs of the per-call timings are
re-used between calls (they fit the 126 MB L2 only at 10k tokens; the step does not).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from modaltune_b200 import config, factory, ops, synthetic, train_step  # noqa: E402
from modaltune_b200.slide_encoder import DILATED_RATIO, optimal_segment_lengths  # noqa: E402

PEAK_BF16 = 2250e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def stats(ts):
    ts = sorted(ts)
    return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1], "n": len(ts)}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def alternate(fns, reps, warm=3):
    for _ in range(warm):
        for f in fns.values():
            f()
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            out[k].append(timed(f))
    return {k: stats(v) for k, v in out.items()}


def attn_inputs(N):
    geom = ops.Geometry.get(N, optimal_segment_lengths(), DILATED_RATIO)
    g = torch.Generator().manual_seed(N)
    qkv = torch.zeros(geom.n_alloc, 2304)
    qkv[:N] = torch.randn(N, 2304, generator=g)
    qkv = qkv.to(torch.bfloat16).cuda()
    gamma, beta = torch.ones(768, device="cuda"), torch.zeros(768, device="cuda")
    dy = torch.randn(N, 768, generator=g).cuda()
    o, l = ops.dilated_attn_fwd(geom, qkv, 3)
    _, _, lse, m, r = ops.dilated_merge_ln_fwd(geom, o, l, gamma, beta)
    dattn, delta = ops.dilated_merge_ln_bwd(geom, dy, o, l, gamma, m, r)
    return geom, qkv, dattn, lse, delta


def attention(N, reps):
    geom, qkv, dattn, lse, delta = attn_inputs(N)
    calls = {f"impl{i}": (lambda i=i: ops.dilated_attn_bwd(geom, qkv, dattn, lse, delta, i)) for i in (2, 4)}
    res = {"per_call": alternate(calls, reps)}
    # kernel times of impl 4 in a profiled run of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            calls["impl4"]()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        if "dilated_bwd" in ev.key or "memset" in ev.key.lower():
            kern[ev.key] = {"total_ms": ev.device_time_total / 1e3 / reps, "launches_per_call": ev.count / reps}
    res["impl4_kernels_per_call"] = kern
    dq = [v["total_ms"] for k, v in kern.items() if "dilated_bwd_dq_sm100_kernel" in k]
    if dq:
        flops = 1.5 * geom.flops_fwd
        res["dq_kernel"] = {"ms_per_call": dq[0], "algorithmic_tflops": flops / (dq[0] * 1e-3) / 1e12,
                            "share_of_bf16_peak": flops / (dq[0] * 1e-3) / PEAK_BF16, "flops": flops}
    res["flops_fwd"] = geom.flops_fwd
    return res


def step(tiles, reps):
    dev = torch.device("cuda")
    model = factory.build_model(None, device=dev)
    proj = factory.build_projector(0, dev)
    flat = train_step.FlatGradAllReduce([p for p in model.parameters() if p.requires_grad])
    host, sizes, _ = train_step.pack_host_slide(synthetic.synthetic_slide(tiles, seed=1000))
    static = {k: v.to(dev) for k, v in host.items()}
    pool = torch.cuda.graph_pool_handle()
    steps = {}
    for det in (False, True):
        with config.using(deterministic=det):
            steps[det] = train_step.GraphedStep(model, proj, static, sizes, flat, pool=pool, static=static)

    def run(det):
        with config.using(deterministic=det):
            steps[det]()

    res = alternate({"default": lambda: run(False), "deterministic": lambda: run(True)}, reps)
    res["ratio"] = res["deterministic"]["median_ms"] / res["default"]["median_ms"]
    del steps
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="directory for deterministic_bench.json")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU: there is no CPU fallback"
    out = {"card": card()}
    for N in (10001, 32769):
        out[f"attn_bwd_{N}"] = attention(N, args.steps)
    for tiles in (10000, 32768):
        out[f"step_{tiles}"] = step(tiles, args.steps)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "deterministic_bench.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
