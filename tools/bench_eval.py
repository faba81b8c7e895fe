"""Evaluation throughput (forward only, no_grad, eval mode, bf16) of the full 331-pathway clinical model, three paths in one
process (the card's name and power limit are read in the same run):

  * per-task   -- one eager ``model(...)`` call per task token: what the reference's ``evaluate`` / ``get_features`` issue;
  * lockstep   -- eager ``forward_tasks`` (``train_step.multitask_forward``): embedding and gene encoder once, the three
                  passes in lockstep through batched frozen layers;
  * graphed    -- ``train_step.GraphedForwardCache``: the same forward captured per token count and replayed (the time
                  includes the device-to-device copy of the slide into the static inputs).

Workloads: one slide of 10 000 tiles, one of 32 768, and the seeded log-uniform 2k-40k mix of bench.py (12 slides,
random.Random(5)) as one pass over all of them.  Slides live on the device before timing.  Each round runs every path
once, in an order that rotates between rounds; per path the median over the rounds is given with the min / max.

    python tools/bench_eval.py [--rounds 7] [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import random
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from modaltune_b200 import config, factory, train_step  # noqa: E402
from modaltune_b200.synthetic import synthetic_slide  # noqa: E402

DEV = "cuda"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def stats(ts):
    s = sorted(ts)
    return {"median_ms": s[len(s) // 2], "min_ms": s[0], "max_ms": s[-1], "n": len(s)}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_eval measures on the GPU; there is no CPU fallback"
    info = card()
    print(json.dumps({"card": info}), flush=True)
    model = factory.build_model(None, clinical=True, device=DEV)
    eye = torch.eye(train_step.NUM_TASKS, device=DEV)
    rnd = random.Random(5)
    mix = [int(math.exp(rnd.uniform(math.log(2000), math.log(40000)))) for _ in range(12)]
    workloads = {"10k": [10000], "32k": [32768], "mix_2k_40k": mix}
    results = {}
    with config.using(mode="bf16"), torch.no_grad():
        for name, counts in workloads.items():
            host = [synthetic_slide(n, seed=1000 + i) for i, n in enumerate(counts)]
            packed = [train_step.pack_host_slide(s)[0] for s in host]
            sizes = train_step.pack_host_slide(host[0], pin=False)[1]
            dev_packed = [{k: v.to(DEV) for k, v in p.items()} for p in packed]
            slides = [train_step.unpack_slide(p, sizes) for p in dev_packed]
            cache = train_step.GraphedForwardCache(model, sizes, max_tiles=max(counts))

            def per_task():
                for s in slides:
                    for t in range(train_step.NUM_TASKS):
                        model(x=s["x"], coords=s["coords"], genes=s["genes"], clinical=s["clinical"], task_token=eye[t])

            def lockstep():
                for s in slides:
                    train_step.multitask_forward(model, s)

            def graphed():
                for p in dev_packed:
                    cache(p)

            paths = {"per_task_eager": per_task, "lockstep_eager": lockstep, "graphed": graphed}
            for fn in paths.values():      # warm-up: module loads, library algorithm choice, one capture per shape
                fn()
                fn()
            # the three paths agree (lockstep and graphed bitwise; per-task runs the per-pass forward of the same model)
            s0 = slides[-1]
            ref = torch.cat([model(x=s0["x"], coords=s0["coords"], genes=s0["genes"], clinical=s0["clinical"],
                                   task_token=eye[t]) for t in range(train_step.NUM_TASKS)], 0)
            lk = train_step.multitask_forward(model, s0)
            gr = cache(dev_packed[-1]).clone()
            agree = {"lockstep_vs_per_task_equal": bool(torch.equal(lk, ref)),
                     "graphed_vs_lockstep_equal": bool(torch.equal(gr, lk))}
            times = {k: [] for k in paths}
            names = list(paths)
            for r in range(args.rounds):
                for k in names[r % 3:] + names[:r % 3]:
                    times[k].append(timed(paths[k]))
            rec = {"tiles": counts, "slides": len(counts), **agree}
            for k in names:
                st = stats(times[k])
                st["slides_per_s"] = len(counts) / (st["median_ms"] / 1e3)
                st["ms_per_slide"] = st["median_ms"] / len(counts)
                rec[k] = st
            rec["speedup_graphed_vs_per_task"] = rec["per_task_eager"]["median_ms"] / rec["graphed"]["median_ms"]
            rec["speedup_lockstep_vs_per_task"] = rec["per_task_eager"]["median_ms"] / rec["lockstep_eager"]["median_ms"]
            results[name] = rec
            print(json.dumps({name: rec}), flush=True)
            del cache, slides, dev_packed
            torch.cuda.empty_cache()
    out = {"card": info, "results": results}
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_eval.json"), "w") as f:
            json.dump(out, f, indent=1)
    for name, rec in results.items():
        print(f"{name:>11}: " + "  ".join(
            f"{k} {rec[k]['ms_per_slide']:.2f} ms/slide ({rec[k]['min_ms'] / rec['slides']:.2f}-"
            f"{rec[k]['max_ms'] / rec['slides']:.2f}), {rec[k]['slides_per_s']:.1f} slides/s"
            for k in ("per_task_eager", "lockstep_eager", "graphed")))


if __name__ == "__main__":
    main()
