#!/usr/bin/env python
"""Benchmark of the ModalTune-GigaPath fine-tuning hot path (BASELINE.json: slides/s fwd+bwd at 10k tiles).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--tiles L] [--mode bf16|fp32]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one slide through the reference's training step: 3 task passes forward, the KL-distillation loss, one backward
(`train_modaltune.py:156-179, 218-235`), plus the data-parallel all-reduce of the trainable gradients when N > 1.  Every
rank processes its own slides (weak scaling, no data-path collective).  Prints ONE JSON line on rank 0.

* ``value``: device-resident slides/s (inputs already in HBM), CUDA events, max over ranks.
* ``e2e``: the same step driven from pinned HOST buffers through the module API, H2D copy of the slide and D2H read of
  loss / logits inside the timed region (every step copies its slide; the copy of slide i + 1 is issued on a copy stream
  while step i runs, ``GraphedStep.prefetch``; the loss / logits of step i are copied to pinned memory behind the step
  and read by the host after step i + 1 has been launched, ``GraphedStep.read_back_async``: every step's result is
  read, none of them stalls the GPU).
* ``roofline``: the dilated-attention backward kernel (the dominant kernel), timed live with CUDA events on its stream
  inside the timed region; algorithmic FLOPs = 2.5 * 4*d*sum c^2 per launch (SURVEY.md §8d) against the measured bf16
  tensor peak of MEASURED_PEAKS.json.
* ``cpu_baseline`` / ``--impl reference``: the oracle port of the reference's CPU arithmetic (the reference is pure
  Python and has no CPU attention of its own) on the host cores: ``cpu_baseline`` = SURVEY.md 8(d)'s C1 protocol (COMPLETE
  oracle training steps at 1 024 tiles, 1 warm-up + 3 timed, median); ``--impl reference`` = ``--steps`` complete oracle
  training steps at the bench tile count (fewer only under an explicit ``--cpu-budget``), reporting the true ``steps``
  it ran (never a scaled figure).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tiles", type=int, default=10000)
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--attn", default="auto", choices=["auto", "simt", "sm100"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=None,
                    help="cap on the seconds of oracle steps the reference arm times (default: no cap, all --steps run)")
    ap.add_argument("--no-extras", action="store_true", help="skip the comparator / 32k / train-mode sub-records")
    ap.add_argument("--no-graph", action="store_true", help="issue every step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (loss, logits, gradients) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU step (--impl ours)")
    return args


UNIT = "slides/s"
# gradient elements --dump-outputs writes: a fixed seeded sample, 16 MB of the 135 MB fp32 gradient of the full model
DUMP_GRAD_SAMPLE = 1 << 22
# DRAM bytes of ONE launch of the default backward attention kernel at 10 001 tokens, from the committed `ncu --set full`
# capture (profiles/r2_ncu_attention.txt)
NCU_TRAFFIC_BWD = 243.571712e6 + 96.210176e6


def metric_name(tiles: int) -> str:
    return f"slides/s fwd+bwd, GigaPath+ModalTune {tiles // 1000}k tiles" if tiles % 1000 == 0 else \
        f"slides/s fwd+bwd, GigaPath+ModalTune {tiles} tiles"


def baseline_config_name(tiles: int) -> str:
    return {1024: "BASELINE.json configs[0]", 10000: "BASELINE.json configs[1]",
            32768: "BASELINE.json configs[2] slide size"}.get(tiles, "custom tile count (not a BASELINE.json config)")


def workload_config(args, world):
    return {
        "workload": f"ModalTune-GigaPath (LongNet 12L/768d/16h dilated attention + Modal Adapter), synthetic "
                    f"{args.tiles}-tile slides + 331 pathway tokens + clinical + text-task embeddings, 3 task passes "
                    f"fwd + KL-distillation loss + bwd per slide ({baseline_config_name(args.tiles)})",
        "tiles": args.tiles, "tokens": args.tiles + 1, "modal_tokens": 66, "task_passes": 3,
        "slides_per_step_per_gpu": 1, "parallelism": f"slide-sharded dp{world}",
        "l2": "working set per step (several GB of saved activations) exceeds the 126 MB L2; no explicit flush",
    }


def dump_outputs(out_dir: str, loss, logits, params) -> None:
    """``--dump-outputs``: what a caller of the step receives, as .npy files that two builds can be compared on.
    ``loss`` (float32 scalar), ``logits`` (float32 [3, 256]), ``grad_norms`` (float64, the L2 norm of every trainable
    parameter's gradient in ``named_parameters`` order) and ``grad_sample`` (float32: the flat gradient vector, in the same
    order, at ``DUMP_GRAD_SAMPLE`` positions drawn with a fixed seed; all of it when it is shorter)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    grads = [(p.grad if p.grad is not None else torch.zeros_like(p)).detach().float().reshape(-1) for p in params]
    flat = torch.cat(grads)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_GRAD_SAMPLE].sort().values
    arrays = {"loss": loss.detach().float().reshape(()), "logits": logits.detach().float(),
              "grad_norms": torch.stack([g.double().norm() for g in grads]), "grad_sample": flat[idx.to(flat.device)]}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: COMPLETE training steps of the oracle port (3 task passes forward + KL loss + backward, 331 pathways)
# ---------------------------------------------------------------------------------------------------------------------
class CpuStep:
    """One slide step of the reference's CPU arithmetic: ``oracle.training_step`` + backward on all host threads, fp32,
    same seeded weights / synthetic slide generator as the GPU arm.  The reference itself is pure Python and does not
    travel to the GPU box (and has no CPU attention of its own, flash_attention.py:143-146), so the arm is the oracle
    port (``kind: "port"``), pinned to the reference by tests/golden."""

    def __init__(self, tiles: int):
        from modaltune_b200 import factory, synthetic
        from oracle import modaltune_oracle as O

        torch.set_num_threads(os.cpu_count() or 1)
        self.O, self.tiles = O, tiles
        # above ~2k tiles the dense attention probabilities of 36 layer passes (5 GB per layer at 10k tiles) cannot
        # stay alive for the backward on any host: every encoder layer is recomputed in the backward, the reference's
        # own ``checkpoint_activations`` option (TS/architecture/encoder.py:317-319).  Same arithmetic, ~1.3x the time.
        self.checkpoint = tiles > 2048
        model = factory.build_model(None)
        self.sd = {k: v.detach().clone().requires_grad_(v.requires_grad) for k, v in model.named_parameters()}
        self.proj_sd = synthetic.seeded_projector_state(0)
        self.table = O.sincos_table()
        self.slides = [synthetic.synthetic_slide(tiles, seed=1000 + i) for i in range(2)]
        # untimed one-off costs (thread pool, allocator, autograd / MKL first touches: ~15 s on the first call) are paid
        # on a tiny 256-tile step, so that even a single timed step is a warm measurement
        tiny = synthetic.synthetic_slide(256, seed=999)
        self._run(tiny)

    def _run(self, s):
        genes = [s["genes"][j] for j in range(len(s["genes"]))]
        for v in self.sd.values():
            v.grad = None
        loss, _ = self.O.training_step(self.sd, self.proj_sd, s["x"][0], s["coords"][0], genes, s["clinical"], s["text"],
                                       table=self.table, checkpoint_layers=self.checkpoint)
        loss.backward()

    def __call__(self, i: int = 0) -> float:
        t0 = time.perf_counter()
        self._run(self.slides[i % len(self.slides)])
        return time.perf_counter() - t0


CPU_ARM_CACHE = os.path.join(os.environ.get("TMPDIR", "/tmp"), "modaltune_b200_cpu_reference_arm.json")


def cpu_baseline(tiles: int):
    """``cpu_baseline`` of the GPU arm.  A complete oracle step at 10k tiles takes minutes of host time, too long for the
    default run, so: (1) SURVEY.md 8(d)'s C1 protocol is always measured here (full oracle step at 1 024 tiles,
    1 warm-up + 3 timed, median); (2) when ``bench.py --impl reference`` has run on THIS box (the driver runs it first),
    its measured full-step figure at the bench tile count is reported as ``value``; otherwise ``value`` is the C1 figure
    and ``sample`` says that it is the 1 024-tile workload.  Nothing is extrapolated."""
    c1 = CpuStep(1024)
    c1(0)
    ts = sorted(c1(i) for i in range(3))
    c1_rec = {"value": 1.0 / ts[1], "unit": UNIT, "tiles": 1024, "seconds_per_step": ts[1], "reps": 3, "warmup": 1,
              "protocol": "SURVEY.md 8(d): full oracle step at 1 024 tiles (BASELINE.json configs[0]), median of 3"}
    cached = None
    try:
        with open(CPU_ARM_CACHE) as f:
            cached = json.load(f)
        if cached.get("tiles") != tiles or time.time() - cached.get("when", 0) > 6 * 3600:
            cached = None
    except Exception:
        cached = None
    if cached is not None:
        return {"value": cached["value"], "unit": UNIT, "cores": cached["cores"], "kind": "port",
                "sample": "measured by `bench.py --impl reference` on this box "
                          f"{time.time() - cached['when']:.0f} s earlier: " + cached["sample"], "c1": c1_rec}
    return {"value": c1_rec["value"], "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
            "sample": f"oracle (CPU restatement of the reference, fp32, torch {torch.get_num_threads()} threads): complete "
                      f"training steps (3 task passes fwd + KL loss + bwd, 331 pathways) at 1 024 tiles (configs[0]), "
                      f"1 warm-up + 3 timed, median {ts[1]:.1f} s.  NOT the {tiles}-tile workload of this line: the "
                      f"full-size CPU figure comes from `bench.py --impl reference` ({tiles} tiles, minutes per step)",
            "c1": c1_rec}


def run_reference(args):
    """``--impl reference``: ``--steps`` complete oracle training steps at the bench tile count on the host cores, after
    one warm-up step when ``--warmup`` > 0.  A step takes about a minute at 10k tiles: ``--cpu-budget S`` caps the run
    at as many steps as fit S seconds (at least one).  Either way the TRUE ``steps`` / ``warmup`` it ran and the measured
    mean are reported, never a scaled figure."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = float("inf") if args.cpu_budget is None else args.cpu_budget
    step = CpuStep(args.tiles)
    t_first = step(0)
    warm = 1 if (args.warmup > 0 and 3.0 * t_first < budget) else 0
    ts = [] if warm else [t_first]
    spent = t_first
    i = 1
    while len(ts) < args.steps and (not ts or spent + ts[-1] < budget):
        ts.append(step(i))
        spent += ts[-1]
        i += 1
    t = sum(ts) / len(ts)
    value = 1.0 / t
    line = {
        "impl": "reference", "metric": metric_name(args.tiles), "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(ts), "warmup": warm, "requested_steps": args.steps, "requested_warmup": args.warmup,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                         "sample": f"{len(ts)} complete oracle training steps (3 task passes fwd + KL loss + bwd, 331 "
                                   f"pathways{', every encoder layer recomputed in the backward (activation checkpointing)' if step.checkpoint else ''}) "
                                   f"at {args.tiles} tiles, {torch.get_num_threads()} threads, "
                                   f"{'1 full warm-up step' if warm else 'warm-up = one untimed 256-tile step'}; steps in seconds: "
                                   f"{[round(x, 1) for x in ts]}; {len(ts)} of {args.steps} requested steps"
                                   f"{'' if args.cpu_budget is None else f' under the {args.cpu_budget:.0f} s budget'}; the "
                                   f"reference is pure Python with no CPU attention kernel of its own "
                                   f"(flash_attn_func is None on CPU), so the arm is the oracle port pinned by tests/golden"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    try:
        with open(CPU_ARM_CACHE, "w") as f:
            json.dump({"tiles": args.tiles, "value": value, "cores": os.cpu_count(), "when": time.time(),
                       "sample": line["cpu_baseline"]["sample"]}, f)
    except OSError:
        pass
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# extra records of the GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def extra_records(args, model, proj, flat, dev, world, rank, timed, barrier):
    """Sub-records next to the headline (never part of `value`): (1) BASELINE config 3's slide size (32 768 tiles, every
    LongNet branch active) through the same graph-replay step; (2) BASELINE config 5: a seeded log-uniform 2k-40k mix,
    assigned to the ranks by `packing.pack_slides` (estimated cost, LPT) and stepped eagerly (one CUDA graph per token
    count cannot serve arbitrary lengths), measured per-rank makespan against the cost model and against the reference's
    equal-count sharding; (3) the train-mode step (`model.train()`: Dropout / DropPath of the frozen encoder and of the
    adapter active, no sharing across the three task passes) + AdamW, which the reference's loop runs."""
    import math
    import random

    import torch.distributed as dist

    from modaltune_b200 import packing, synthetic, train_step

    out = {}
    # (1) 32 768-tile slides
    try:
        host = train_step.pack_host_slide(synthetic.synthetic_slide(32768, seed=3000 + rank))
        res = {k: v.to(dev) for k, v in host[0].items()}
        g32 = train_step.GraphedStep(model, proj, res, host[1], flat)
        for _ in range(2):
            g32(res)
        ms = timed(lambda i: g32(res), 3)
        out["c3_32k_tiles"] = {"tiles": 32768, "ms_per_step": ms / 3, "slides_per_s": world * 3 / (ms / 1e3), "steps": 3,
                               "n_gpus": world, "execution": "cuda-graph replay", "config": "BASELINE.json configs[2] slide size"}
        del g32, res, host
        torch.cuda.empty_cache()
    except Exception as e:
        out["c3_32k_tiles"] = {"failed": f"{type(e).__name__}: {str(e)[:200]}"}
    # (2) variable tile counts, packed
    try:
        per_gpu = 12
        rnd = random.Random(5)
        counts = [int(math.exp(rnd.uniform(math.log(2000), math.log(40000)))) for _ in range(per_gpu * world)]
        shards, est = packing.pack_slides(counts, world)
        _, est_rr = packing.round_robin(counts, world)
        mine = shards[rank]

        def run_shard(_):
            flat.zero()
            for i in mine:
                slide = train_step.slide_to_device(synthetic.synthetic_slide(counts[i], seed=5000 + i), dev)
                train_step.forward_backward(model, proj, slide)
            flat.all_reduce()

        hosts = [synthetic.synthetic_slide(counts[i], seed=5000 + i) for i in mine]   # generated before the timed region
        train_step.forward_backward(model, proj, train_step.slide_to_device(hosts[0], dev))   # warm the allocator
        flat.zero()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        flat.zero()
        for h in hosts:
            train_step.forward_backward(model, proj, train_step.slide_to_device(h, dev))
        e1.record()
        torch.cuda.synchronize()
        own = torch.tensor([e0.elapsed_time(e1)], device=dev)
        allr = [torch.zeros_like(own) for _ in range(world)]
        if world > 1:
            dist.all_gather(allr, own)
        else:
            allr = [own]
        flat.all_reduce()
        per_rank = [float(t) for t in allr]
        mean = sum(per_rank) / world
        out["c5_variable_tiles"] = {
            "slides": len(counts), "tile_range": [min(counts), max(counts)], "n_gpus": world, "execution": "eager (one shape per slide)",
            "per_rank_ms": per_rank, "makespan_ms": max(per_rank), "measured_imbalance": max(per_rank) / mean - 1.0,
            "slides_per_s": len(counts) / (max(per_rank) / 1e3),
            "cost_model": {"packed_imbalance": est["imbalance"], "equal_count_imbalance": est_rr["imbalance"],
                           "packed_makespan_ms": est["makespan_ms"]},
            "note": "host slides pre-generated; each step copies its slide from pageable host memory (the reference's 331 + 4 copies)",
            "config": "BASELINE.json configs[4] (seeded log-uniform 2k-40k tiles, packed by estimated cost)"}
        try:
            # the same shard through train_step.GraphCache: one captured step per tile count in a shared memory pool.  Epoch 1
            # captures every shape (all misses), epoch 2 revisits the same slides (what training does): all hits.
            packed = [train_step.pack_host_slide(h) for h in hosts]
            cache = train_step.GraphCache(model, proj, flat, packed[0][1], max_tiles=max(counts) + 1)
            accum = []

            def epoch():
                for a in accum:
                    a.zero_()
                for pk in packed:
                    cache(pk[0])
                    bufs = cache.steps[int(pk[0]["x"].shape[-2])].grad_buffers    # consumed before the next replay
                    if not accum:
                        accum.extend(torch.zeros_like(b) for b in bufs)
                    torch._foreach_add_(accum, bufs)

            ep = []
            for _ in range(2):
                torch.cuda.synchronize()
                e0.record()
                epoch()
                e1.record()                  # this rank's own work: the exchange below would hide the imbalance
                if world > 1:
                    for a in accum:
                        dist.all_reduce(a)
                torch.cuda.synchronize()
                own = torch.tensor([e0.elapsed_time(e1)], device=dev)
                allr = [torch.zeros_like(own) for _ in range(world)]
                if world > 1:
                    dist.all_gather(allr, own)
                else:
                    allr = [own]
                ep.append([float(t) for t in allr])
            mean2 = sum(ep[1]) / world
            out["c5_variable_tiles"]["graph_cache"] = {
                "execution": "train_step.GraphCache: one captured step per tile count, shared memory pool and input buffers",
                "epoch1_capture_ms": max(ep[0]), "epoch2_replay_per_rank_ms": ep[1], "epoch2_makespan_ms": max(ep[1]),
                "epoch2_measured_imbalance": max(ep[1]) / mean2 - 1.0, "epoch2_slides_per_s": len(counts) / (max(ep[1]) / 1e3),
                "hits": cache.hits, "misses": cache.misses, "distinct_shapes": len(cache.steps)}
            del cache, packed
            accum.clear()
            flat.zero()
            torch.cuda.empty_cache()
        except Exception as e:
            out["c5_variable_tiles"]["graph_cache"] = {"failed": f"{type(e).__name__}: {str(e)[:300]}"}
    except Exception as e:
        out["c5_variable_tiles"] = {"failed": f"{type(e).__name__}: {str(e)[:200]}"}
    # (3) train mode + optimizer
    try:
        host = train_step.pack_host_slide(synthetic.synthetic_slide(args.tiles, seed=4000 + rank))
        slide = train_step.unpack_slide({k: v.to(dev) for k, v in host[0].items()}, host[1])
        opt = torch.optim.AdamW([p for p in model.parameters() if p.requires_grad], lr=1e-6)
        model.train()

        def train_it(_):
            opt.zero_grad()
            train_step.forward_backward(model, proj, slide)
            flat.all_reduce()
            opt.step()

        for _ in range(2):
            train_it(0)
        ms = timed(train_it, 3)
        out["train_mode"] = {"tiles": args.tiles, "ms_per_step": ms / 3, "slides_per_s": world * 3 / (ms / 1e3), "steps": 3,
                             "execution": "eager, model.train(): Dropout(0.25) / DropPath in the frozen encoder and the adapter, "
                                          "fresh masks in each of the three task passes, AdamW step included"}
        # the same step captured in a CUDA graph (the Philox seeds and DropPath factors are drawn on the device inside
        # the graph, so every replay has fresh masks) + AdamW on the gradients the replay hands back
        gtr = train_step.GraphedStep(model, proj, {k: v.to(dev) for k, v in host[0].items()}, host[1], flat)

        def train_graph(_):
            opt.zero_grad()
            gtr()
            opt.step()

        for _ in range(2):
            train_graph(0)
        ms = timed(train_graph, 5)
        out["train_mode"]["graph_replay"] = {"ms_per_step": ms / 5, "slides_per_s": world * 5 / (ms / 1e3), "steps": 5}
        del gtr
        model.eval()
        flat.zero()
    except Exception as e:
        model.eval()
        out["train_mode"] = {"failed": f"{type(e).__name__}: {str(e)[:200]}"}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist

    from modaltune_b200 import _lib, config, factory, ops, synthetic, train_step

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path in modaltune_b200)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    config.set_mode(args.mode)
    config.set_attn_impl(args.attn)

    model = factory.build_model(None, device=dev)          # full 331-pathway ModalTune-GigaPath, seeded random init
    proj = factory.build_projector(0, dev)
    flat = train_step.FlatGradAllReduce([p for p in model.parameters() if p.requires_grad])
    n_slides = 2
    hosts = [train_step.pack_host_slide(synthetic.synthetic_slide(args.tiles, seed=1000 + rank * 100 + i))
             for i in range(n_slides)]
    sizes, h2d_bytes = hosts[0][1], hosts[0][2]
    resident = [{k: v.to(dev) for k, v in h.items()} for h, _, _ in hosts]
    geom = ops.Geometry.get(args.tiles + 1, model.segment_lengths, (1, 2, 4, 8, 16))

    def eager_step(packed):
        flat.zero()
        loss, logits = train_step.forward_backward(model, proj, train_step.unpack_slide(packed, sizes))
        flat.all_reduce()
        return loss, logits

    graphed = None if args.no_graph else train_step.GraphedStep(model, proj, resident[0], sizes, flat)
    step = eager_step if graphed is None else graphed

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(run, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            run(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    # ---- warm-up -------------------------------------------------------------------------------------------------
    for i in range(max(args.warmup, 3)):
        step(resident[i % n_slides])
    torch.cuda.synchronize()

    # ---- device-resident timed region (inputs already in HBM; every step takes the other slide) -----------------------
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    launches0 = ops.launch_count
    last = [None]

    def resident_step(i):
        last[0] = step(resident[i % n_slides])

    ms = timed(resident_step, args.steps)
    value = world * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        # before the e2e region below replays the graph again and overwrites its outputs
        dump_outputs(args.dump_outputs, *last[0], [p for p in model.parameters() if p.requires_grad])

    # ---- end to end: pinned host -> device, step, loss/logits back to the host ---------------------------------------
    out = {}

    pending = []

    def read(ev, lh, gh):
        ev.synchronize()
        out["loss"], out["logits"] = float(lh), gh.clone()

    def e2e_step(i, last=None):
        h = hosts[i % n_slides][0]
        if graphed is None:
            loss, logits = eager_step({k: v.to(dev, non_blocking=True) for k, v in h.items()})
            out["loss"], out["logits"] = float(loss), logits.float().cpu()   # D2H reads (synchronising, like loss.item())
            return
        graphed(h)
        graphed.prefetch(hosts[(i + 1) % n_slides][0])   # the next slide's H2D copy overlaps this step
        # D2H read of EVERY step's loss / logits, one step late: the copy into pinned memory is queued behind the step,
        # the host waits for it only after the next step has been launched (no GPU idle time around a loss.item())
        pending.append(graphed.read_back_async())
        if len(pending) > 1:
            read(*pending.pop(0))
        if i == (args.steps - 1 if last is None else last):
            read(*pending.pop(0))                        # the last step of the timed region is read inside it

    e2e_step(0, last=0)
    ms_e2e = timed(e2e_step, args.steps)
    e2e_value = world * args.steps / (ms_e2e / 1e3)

    # ---- per-kernel timing + launch count: the same step issued eagerly with CUDA events around the attention kernels -
    for i in range(2):  # the caching allocator needs its blocks back on this stream after the graph capture
        eager_step(resident[i % n_slides])
    ops.kernel_events = {}
    launches0 = ops.launch_count
    ms_eager = timed(lambda i: eager_step(resident[i % n_slides]), args.steps)
    launches = (ops.launch_count - launches0) // args.steps
    events, ops.kernel_events = ops.kernel_events, None
    clk = clocks.stop() if rank == 0 else None

    # ---- extra records (all ranks take part: the steps all-reduce): BASELINE configs 3 and 5, train mode ---------------
    extras = {}
    if not args.no_extras:
        extras = extra_records(args, model, proj, flat, dev, world, rank, timed, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (dilated-attention backward) ------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    else:
        peak, peak_src = 1590.0, "fallback (B200_PROFILING.md)"
    f_fwd, f_bwd = ops.attention_flops(geom)

    def avg_ms(name):
        ev = events.get(name, [])
        return sum(a.elapsed_time(b) for a, b in ev) / max(len(ev), 1), len(ev)

    t_bwd, n_bwd = avg_ms("dilated_attn_bwd")
    t_fwd, n_fwd = avg_ms("dilated_attn_fwd")
    ach_bwd = f_bwd / (t_bwd * 1e-3) / 1e12 if t_bwd > 0 else 0.0
    ach_fwd = f_fwd / (t_fwd * 1e-3) / 1e12 if t_fwd > 0 else 0.0
    # DRAM bytes per launch of the backward kernel from the committed `ncu --set full` capture (read + write); only valid
    # for the configuration that capture was taken on
    traffic, traffic_src = None, None
    if args.tiles == 10000 and config.attn_impl("bwd") == 2 and NCU_TRAFFIC_BWD is not None:
        traffic = NCU_TRAFFIC_BWD
        traffic_src = "profiles/r2_ncu_attention.txt (dram__bytes_read.sum + dram__bytes_write.sum, one launch)"
    bwd_names = {0: "simt", 1: "tcgen05", 2: "tcgen05-persistent"}
    fwd_names = {0: "simt", 1: "tcgen05, 128-key tiles", 3: "tcgen05, 48-key tiles, 4 CTAs per SM"}
    roofline = {
        "bound": "tensor", "kernel": f"dilated_attn_bwd[{bwd_names[config.attn_impl('bwd')]}]", "achieved": ach_bwd,
        "peak": peak, "peak_source": peak_src, "unit": "TFLOP/s", "frac": ach_bwd / peak, "traffic": traffic,
        "traffic_source": traffic_src,
        "launch_ms": t_bwd, "launches_timed": n_bwd, "algorithmic_gflop_per_launch": f_bwd / 1e9,
        "share_of_step": t_bwd * n_bwd / args.steps / (ms / args.steps),
        "timing": "CUDA events on the launching stream, eager pass of the same step inside this run",
        "fwd": {"kernel": f"dilated_attn_fwd[{fwd_names[config.attn_impl('fwd')]}]", "achieved": ach_fwd,
                "frac": ach_fwd / peak, "launch_ms": t_fwd, "launches_timed": n_fwd,
                "algorithmic_gflop_per_launch": f_fwd / 1e9, "share_of_step": t_fwd * n_fwd / args.steps / (ms / args.steps)},
    }
    line = {
        "metric": metric_name(args.tiles), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if args.mode == "bf16" else "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": 4 + 3 * 256 * 4, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
        "execution": "eager" if graphed is None else "cuda-graph replay of the captured step (one graph per token count)",
        "eager_ms_per_step": ms_eager / args.steps, "clocks": clk, "roofline": roofline,
        "attention_tflops": {"fwd": ach_fwd, "bwd": ach_bwd},
        "loss": out.get("loss"),
    }
    if extras:
        line["extras"] = extras
    if world == 1 and not args.no_extras:
        # same-box END-TO-END comparator: the unmodified reference modules under fp16 autocast with the installed flash-attn
        # (its real GPU path; staged under oracle/_ref/reference by __graft_entry__.build()), one training step at this size
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_reference_gpu

            line["reference_gpu_path"] = bench_reference_gpu.run(args.tiles, steps=3, warmup=2, dev=dev)
            line["reference_gpu_path"]["speedup_ours_e2e"] = e2e_value / line["reference_gpu_path"]["slides_per_s"]
        except Exception as e:
            line["reference_gpu_path"] = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
        # same-box comparator: the kernel the reference runs (flash_attn_func, FA2 built for sm_100) on its five per-layer
        # shapes at this token count, next to our kernels (tools/bench_fa2_branches.py); library code, comparator only
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_fa2_branches

            line["fa2_comparator"] = bench_fa2_branches.run(args.tiles + 1, reps=5, dev=dev)
        except Exception as e:  # flash-attn missing on the box: say so, the bench line stands
            line["fa2_comparator"] = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args.tiles)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
