"""What the Modal Adapter's attention maps cost on the GPU, in one process (the card's name and power limit are read in the
same run):

  * one mt_cross_attn_probs call (impl 1, the bf16-mode kernel, and impl 0, the fp32-mode kernel) at the adapter's shapes:
    Injector 10 000 x 66 and 32 768 x 66 (tiles over modal tokens), Extractor 66 x 10 000 and 66 x 32 768, prompt
    self-attention 66 x 66; with the bytes the call must write (the [Lq, Lk] fp32 map) over its time;
  * the eager three-task forward (full 331-pathway model, eval, bf16 mode, no autograd) at 10k tiles with and without a
    forward hook on every Modal Adapter attention module, alternated after a warm-up.

    python tools/bench_attn_weights.py [--reps 20] [--out DIR]

Every time is the median of CUDA-event timings with the min / max beside it.  Per-call timings launch the kernel
``--launches`` times between two events and divide (host side included); ``kernel_ms`` is the kernel's device time from
a ``torch.profiler`` run of its own.  Inputs stay in L2 between launches (they are < 30 MB).
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
import torch.nn as nn  # noqa: E402

from modaltune_b200 import config, factory, ops, synthetic, train_step  # noqa: E402

H, E = 12, 192
SHAPES = {"injector_10k": (10000, 66), "injector_32k": (32768, 66), "extractor_10k": (66, 10000),
          "extractor_32k": (66, 32768), "prompt": (66, 66)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def stats(ts):
    ts = sorted(ts)
    return {"median_ms": ts[len(ts) // 2], "min_ms": ts[0], "max_ms": ts[-1], "n": len(ts)}


def timed(fn, n=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def alternate(fns, reps, n=1, warm=3):
    for _ in range(warm):
        for f in fns.values():
            f()
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            out[k].append(timed(f, n))
    return {k: stats(v) for k, v in out.items()}


def kernel(lq, lk, reps, launches):
    g = torch.Generator(device="cuda").manual_seed(lq + lk)
    q = torch.randn(lq, E, device="cuda", generator=g)
    kv = torch.randn(lk, 2 * E, device="cuda", generator=g)
    k = kv[:, :E]
    lse = {i: ops.cross_attn_fwd(q, k, kv[:, E:], H, impl=i)[1] for i in (0, 1)}
    res = alternate({f"impl{i}": (lambda i=i: ops.cross_attn_probs(q, k, lse[i], H, impl=i)) for i in (0, 1)}, reps,
                    n=launches)
    # the per-call times above include the host side of a launch (ctypes, allocation), which exceeds the kernel at
    # these sizes: the kernel's own time comes from a profiled run of its own
    from torch.profiler import ProfilerActivity, profile
    out_bytes = 4 * lq * lk
    for i in (0, 1):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(launches):
                ops.cross_attn_probs(q, k, lse[i], H, impl=i)
            torch.cuda.synchronize()
        ms = sum(ev.device_time_total for ev in prof.key_averages() if "cross_probs" in ev.key) / 1e3 / launches
        res[f"impl{i}"]["kernel_ms"] = ms
        res[f"impl{i}"]["output_GB_per_s"] = out_bytes / (ms * 1e-3) / 1e9
    res["output_bytes"] = out_bytes
    return res


def forward(tiles, reps):
    dev = torch.device("cuda")
    model = factory.build_model(None, device=dev)
    slide = train_step.slide_to_device(synthetic.synthetic_slide(tiles, seed=1000), dev)
    mhas = [m for m in model.modules() if isinstance(m, nn.MultiheadAttention)]
    maps = []

    def run(hooked):
        handles = [m.register_forward_hook(lambda mod, a, out: maps.append(out[1])) for m in mhas] if hooked else []
        with torch.no_grad():
            train_step.multitask_forward(model, slide)
        for h in handles:
            h.remove()
        n = len(maps)
        maps.clear()
        return n

    with config.using(mode="bf16"):
        assert run(True) == len(mhas) * train_step.NUM_TASKS
        res = alternate({"no_hooks": lambda: run(False), "hooks_on_all_attention": lambda: run(True)}, reps)
    res["ratio"] = res["hooks_on_all_attention"]["median_ms"] / res["no_hooks"]["median_ms"]
    res["hooked_modules"] = len(mhas)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--launches", type=int, default=50, help="kernel launches between two events")
    ap.add_argument("--out", default=None, help="directory for attn_weights_bench.json")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU: there is no CPU fallback"
    out = {"card": card()}
    for name, (lq, lk) in SHAPES.items():
        out[f"kernel_{name}"] = kernel(lq, lk, args.reps, args.launches)
    out["forward_3_tasks_10k"] = forward(10000, args.reps)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "attn_weights_bench.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
