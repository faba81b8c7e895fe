"""One ModalTune training step on the hot path: three task passes forward, the KL-distillation loss, one backward.

Host-side mirror of ``MILTextGeneTrainer_multitask.multitask_forward`` + the loss of ``train_one_epoch``
(``train_modaltune.py:156-179, 211-235``) and of the frozen random text projector (``:44-59``); the data-parallel
gradient exchange replaces DDP's bucketed all-reduce (``utils/base_trainer.py:205-211``) with ONE NCCL all-reduce over
a flat buffer of the trainable gradients (SURVEY.md §8e).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

NUM_TASKS = 3          # utils/constants.py:45-49: 0 General, 1 Diagnosis, 2 Survival
TEXT_ROWS = (0, 1, 3)  # train_modaltune.py:230-233


class Projection_layer(nn.Module):
    """Frozen random text projector (train_modaltune.py:44-59): Conv1x1(512->256), LN([256,1,1]), ReLU, Conv1x1."""

    def __init__(self, in_dim: int = 512, out_dim: int = 256):
        super().__init__()
        self.conv1 = nn.Sequential(nn.Conv2d(in_dim, out_dim, 1), nn.LayerNorm([out_dim, 1, 1]), nn.ReLU(),
                                   nn.Conv2d(out_dim, out_dim, 1))
        for p in self.parameters():
            p.requires_grad = False

    def forward(self, x):
        return self.conv1(x.unsqueeze(-1).unsqueeze(-1)).squeeze(-1).squeeze(-1)


def text_targets(projector: nn.Module, text: torch.Tensor) -> torch.Tensor:
    t = projector(text.float())
    return t / t.norm(dim=-1, keepdim=True)


def multitask_forward(model, slide: Dict, task_ids: Sequence[int] = (0, 1, 2), split_grads: bool = False) -> torch.Tensor:
    """[len(task_ids), 256] task-conditioned embeddings (train_modaltune.py:156-179).  ``split_grads``: see
    ``LongNetGeneAdapter.forward_tasks`` (only for callers that collect the per-pass gradients, ``forward_backward``)."""
    eye = torch.eye(NUM_TASKS, device=slide["x"].device)
    clinical = slide.get("clinical") if getattr(model, "_HAS_CLINICAL", False) else None
    if hasattr(model, "forward_tasks"):
        return model.forward_tasks(slide["x"], slide["coords"], slide["genes"], clinical, [eye[t] for t in task_ids],
                                   split_grads=split_grads)
    outs = []
    for t in task_ids:
        kw = {"clinical": clinical} if clinical is not None else {}
        outs.append(model(x=slide["x"], coords=slide["coords"], genes=slide["genes"], task_token=eye[t], **kw))
    return torch.cat(outs, 0)


def distill_loss(logits: torch.Tensor, text_proj: torch.Tensor) -> torch.Tensor:
    """10 * KLDiv_sum(log_softmax(z/|z|), softmax(t[[0,1,3]]))   (train_modaltune.py:225-233)."""
    z = logits.float()
    z = z / z.norm(dim=-1, keepdim=True)
    tgt = F.softmax(torch.stack([text_proj[r] for r in TEXT_ROWS], 0), dim=1)  # no host index tensor (graph capture)
    return F.kl_div(F.log_softmax(z, dim=1), tgt, reduction="sum") * 10.0


def forward_backward(model, projector, slide: Dict):
    """One slide step: returns (loss, logits).  Gradients are left in ``p.grad`` of the trainable parameters.

    The gradients are taken with ``torch.autograd.grad`` and assigned, not accumulated by ``loss.backward()``: an
    AccumulateGrad node remembers the CUDA stream of the step that created it, and a node kept alive from an earlier
    (eager, default-stream) step silently breaks a later multi-stream CUDA-graph capture of the same model."""
    logits = multitask_forward(model, slide, split_grads=True)
    loss = distill_loss(logits, text_targets(projector, slide["text"]))
    named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
    params = [p for _, p in named]
    aliases = getattr(model, "_pass_aliases", None)
    if aliases:
        # one gradient per (parameter, task pass): the passes read the parameters through their own leaf aliases, so the
        # engine does not sum their contributions one tiny kernel at a time; two multi-tensor adds do it here
        targets, owner = [], []
        for i, (n, p) in enumerate(named):
            for t in ([a[n] for a in aliases] if n in aliases[0] else [p]):
                targets.append(t)
                owner.append(i)
        model._pass_aliases = None
        raw = torch.autograd.grad(loss, targets, allow_unused=True)
        if hasattr(model, "join_pass_streams"):
            model.join_pass_streams()
        per = [[] for _ in params]
        for i, g in zip(owner, raw):
            if g is not None:
                per[i].append(g)
        grads = [gs[0] if gs else None for gs in per]
        depth = max((len(gs) for gs in per), default=0)
        for d in range(1, depth):      # out of place: a gradient the engine returns may alias another one
            idx = [i for i, gs in enumerate(per) if len(gs) > d]
            if idx:
                for i, g in zip(idx, torch._foreach_add([grads[i] for i in idx], [per[i][d] for i in idx])):
                    grads[i] = g
    else:
        grads = torch.autograd.grad(loss, params, allow_unused=True)
        if hasattr(model, "join_pass_streams"):
            model.join_pass_streams()     # the backward of a task pass runs on the stream of its forward
    for p, g in zip(params, grads):
        if g is not None:
            p.grad = g if p.grad is None else p.grad + g
    return loss.detach(), logits.detach()


def slide_to_device(slide: Dict, device, non_blocking: bool = True) -> Dict:
    out = {}
    for k, v in slide.items():
        if isinstance(v, dict):
            out[k] = {kk: vv.to(device, non_blocking=non_blocking) for kk, vv in v.items()}
        else:
            out[k] = v.to(device, non_blocking=non_blocking)
    return out


class FlatGradAllReduce:
    """Data-parallel gradient exchange: the gradients of all trainable parameters are gathered into ONE contiguous fp32
    buffer (one cat kernel), all-reduced with a single NCCL call (sum, then / world) and handed back as views, so
    ``p.grad`` of every parameter aliases the reduced buffer.  Replaces DDP's 25 MB-bucket all-reduces
    (utils/base_trainer.py:205-211).  ``zero()`` drops the gradients (set-to-none): the next backward then WRITES
    instead of accumulating, which saves one tiny add kernel per parameter (1 500+ per step for the gene encoder)."""

    def __init__(self, params: Sequence[torch.nn.Parameter]):
        self.params = [p for p in params if p.requires_grad]
        assert all(p.dtype == torch.float32 for p in self.params)
        self.numel = sum(p.numel() for p in self.params)
        self.flat = None

    def zero(self):
        for p in self.params:
            p.grad = None

    def gather(self):
        """Flatten the current gradients into one buffer and re-point ``p.grad`` at its slices."""
        dev = self.params[0].device
        parts = [(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in self.params]
        self.flat = torch.cat(parts)
        off = 0
        for p in self.params:
            p.grad = self.flat[off:off + p.numel()].view_as(p)
            off += p.numel()
        return self.flat

    def _stacked_groups(self):
        """Gradients that autograd delivers as views of one contiguous fp32 tensor which they tile completely (the
        per-pathway SNN parameters of the gene encoder, evaluated as grouped GEMMs over ``cat`` / ``stack``-ed weights):
        -> ([(base, [param index, ...]), ...], [indices of all other parameters])."""
        groups: Dict[int, list] = {}
        order: List[int] = []
        plain: List[int] = []
        for i, p in enumerate(self.params):
            g = p.grad
            base = g._base if g is not None else None
            if base is not None and base.dtype == torch.float32 and base.is_contiguous():
                if id(base) not in groups:
                    groups[id(base)] = [base, 0, []]
                    order.append(id(base))
                groups[id(base)][1] += g.numel()
                groups[id(base)][2].append(i)
            else:
                plain.append(i)
        stacked = []
        for k in order:
            base, covered, members = groups[k]
            if covered == base.numel() and len(members) > 1:
                stacked.append((base, members))
            else:
                plain.extend(members)
        plain.sort()
        return stacked, plain

    def _dense_group(self, base: torch.Tensor, members: List[int]) -> torch.Tensor:
        """The gradients of one stacked group in PARAMETER layout.  When every view is already laid out like its parameter
        (slices of a ``stack``) the base itself is returned.  Otherwise (the 331 transposed slices of the ``cat``-ed first
        SNN layer) ONE gather kernel writes a buffer of consecutive parameter-layout blocks and ``p.grad`` is re-pointed
        at them: an optimizer's multi-tensor path wants gradients with the strides of their parameters, and producing
        them one transposing copy per pathway is what the flat gather of round 1 spent most of its time on.  The gather
        index depends on the model only and is cached."""
        grads = [self.params[i].grad for i in members]
        if all(g.is_contiguous() for g in grads):
            return base
        key = (tuple(base.shape),) + tuple((g.storage_offset() - base.storage_offset(), tuple(g.shape), tuple(g.stride()))
                                           for g in grads)
        cache = self.__dict__.setdefault("_gather_index", {})
        if key not in cache:
            idx = []
            for off, shape, stride in key[1:]:
                t = torch.full(shape, off, dtype=torch.int64)
                for d, (n, st) in enumerate(zip(shape, stride)):
                    view = [1] * len(shape)
                    view[d] = n
                    t = t + (torch.arange(n, dtype=torch.int64) * st).view(view)
                idx.append(t.reshape(-1))
            cache[key] = torch.cat(idx).to(base.device)
        dense = base.reshape(-1).index_select(0, cache[key])
        off = 0
        for i in members:
            p = self.params[i]
            p.grad = dense[off:off + p.numel()].view_as(p)
            off += p.numel()
        return dense

    def densify(self) -> None:
        """Make every ``p.grad`` dense in its parameter's layout (one gather kernel per stacked group that needs it);
        what a single-rank step does instead of ``gather_buffers``."""
        stacked, _ = self._stacked_groups()
        for base, members in stacked:
            self._dense_group(base, members)
        # stragglers: strided gradients that are not views any more (train mode: the engine sums the three passes'
        # transposed slices into a tensor that keeps their strides).  One copy each -- a single gradient without the
        # strides of its parameter sends an optimizer's WHOLE multi-tensor update down the one-tensor-at-a-time path
        # (measured: AdamW 5 -> 15 ms per step)
        for p in self.params:
            if p.grad is not None and not p.grad.is_contiguous():
                p.grad = p.grad.contiguous()

    def gather_buffers(self) -> List[torch.Tensor]:
        """A few contiguous fp32 buffers that together hold every gradient exactly once, WITHOUT flattening the 1 324
        per-pathway gradients of the gene encoder one by one (331 transposing copies and most of a ~50-launch ``cat``
        per step in round 1): each stacked group is exchanged as its base tensor, or as one gathered parameter-layout
        buffer (``_dense_group``), and ``p.grad`` aliases it.  The remaining gradients go into one small flat buffer.
        The layout is a function of the model only, so every rank builds the same list."""
        stacked, plain = self._stacked_groups()
        bufs = [self._dense_group(base, members) for base, members in stacked]
        parts = [(self.params[i].grad if self.params[i].grad is not None else torch.zeros_like(self.params[i])).reshape(-1)
                 for i in plain]
        small = torch.cat(parts) if parts else torch.zeros(0, device=self.params[0].device)
        off = 0
        for i in plain:
            p = self.params[i]
            p.grad = small[off:off + p.numel()].view_as(p)
            off += p.numel()
        self.buffers = [small] + bufs
        return self.buffers

    def all_reduce(self):
        import torch.distributed as dist

        flat = self.gather()
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM)
            flat.div_(dist.get_world_size())
        return flat


# ---------------------------------------------------------------------------------------------------------------------
# CUDA-graph step
# ---------------------------------------------------------------------------------------------------------------------
def pack_host_slide(slide: Dict, pin: bool = True):
    """Host staging of one case: x, coords, clinical, text plus the 331 pathway vectors packed into ONE buffer (one H2D
    copy instead of the reference's 331, train_modaltune.py:205-208).  Returns (tensors, pathway sizes, bytes)."""
    sizes = [slide["genes"][i].shape[1] for i in range(len(slide["genes"]))]
    host = {"x": slide["x"].float(), "coords": slide["coords"].float(),
            "genes_flat": torch.cat([slide["genes"][i].reshape(-1) for i in range(len(sizes))]).float(),
            "clinical": slide["clinical"].float(), "text": slide["text"].float()}
    host = {k: (v.contiguous().pin_memory() if pin and torch.cuda.is_available() else v.contiguous())
            for k, v in host.items()}
    return host, sizes, sum(v.numel() * v.element_size() for v in host.values())


def unpack_slide(packed: Dict, sizes: Sequence[int]) -> Dict:
    """Views of a packed slide in the layout the model takes (``genes`` as a dict of [1, n_i] views)."""
    d = {k: v for k, v in packed.items() if k != "genes_flat"}
    d["genes"] = {i: p.unsqueeze(0) for i, p in enumerate(torch.split(packed["genes_flat"], list(sizes)))}
    return d


class GraphedStep:
    """forward (3 task passes) + loss + backward + gradient flattening of ONE slide shape captured in a CUDA graph.

    A step launches ~5 000 kernels, most of them tiny (gene encoder, modal-token side of the adapter, autograd glue);
    issued eagerly from Python the step is CPU-bound.  Captured once per token count, a step is one
    ``cudaGraphLaunch``: the inputs are copied into static device buffers, the graph is replayed, the single NCCL
    all-reduce of the flat gradient buffer runs after it.  Gradients live in ``flat.flat`` / ``p.grad`` views."""

    def __init__(self, model, projector, packed_example: Dict, sizes: Sequence[int], flat: FlatGradAllReduce,
                 warmup: int = 3, pool=None, static: Optional[Dict] = None, flatten: Optional[bool] = None):
        """``pool``: a ``torch.cuda.graph_pool_handle()`` shared with other captured steps that are never replayed
        concurrently (``GraphCache``); ``static``: pre-allocated device input buffers of the captured shapes (views of a
        buffer shared by such steps) instead of private copies; ``flatten``: gather the gradients into ONE flat buffer
        inside the graph into the few contiguous buffers the all-reduce runs on (``FlatGradAllReduce.gather_buffers``).
        Default: only when there is more than one rank -- with a single rank nothing is exchanged; ``grads`` concatenates
        on demand either way."""
        import torch.distributed as dist
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        self._flatten = multi if flatten is None else bool(flatten)
        self.model, self.projector, self.flat, self.sizes = model, projector, flat, list(sizes)
        dev = next(model.parameters()).device
        if static is None:
            self.static = {k: v.to(dev).clone() for k, v in packed_example.items()}
        else:
            self.static = static
            for k, v in self.static.items():
                assert v.shape == packed_example[k].shape and v.device == dev
                v.copy_(packed_example[k], non_blocking=True)
        self._copy_stream, self._staging, self._staged_for = None, None, None
        self._warmup, self._pool = warmup, pool
        self._capture()

    def _capture_signature(self):
        """What the captured kernels depend on besides the inputs: the deterministic switch (a graph captured with the
        fast backward must never replay as deterministic, nor the other way round) and the frozen weights."""
        from . import config
        return config.deterministic(), self._frozen_signature()

    def _frozen_signature(self):
        """Identity + version of every frozen parameter the captured kernels read through derived copies
        (``ops.FrozenLayerWeights``): a ``load_state_dict`` / in-place edit after capture changes it."""
        return tuple((p.data_ptr(), p._version) for p in self.model.parameters() if not p.requires_grad)

    def _capture(self):
        model, projector, flat, warmup = self.model, self.projector, self.flat, self._warmup
        slide = unpack_slide(self.static, self.sizes)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                flat.zero()
                forward_backward(model, projector, slide)
                flat.densify()     # also builds the (cached) gather indices outside the capture
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        flat.zero()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, pool=self._pool):
            self.loss, self.logits = forward_backward(model, projector, slide)
            if self._flatten:
                self._bufs = flat.gather_buffers()
            else:
                self._bufs = None
                flat.densify()     # gradients in parameter layout: the optimizer's multi-tensor path
        # views of the captured flat buffer, handed back to ``p.grad`` after every replay
        self._grad_views = [p.grad for p in flat.params]
        self._signature = self._capture_signature()

    @property
    def grads(self) -> torch.Tensor:
        """The flat fp32 gradient vector of the last replay (the captured buffer, or a concatenation made on demand)."""
        return torch.cat([(g if g is not None else torch.zeros_like(p)).reshape(-1)
                          for p, g in zip(self.flat.params, self._grad_views)])

    @property
    def grad_buffers(self) -> Optional[List[torch.Tensor]]:
        """The captured contiguous gradient buffers (``FlatGradAllReduce.gather_buffers``; None when captured with
        ``flatten=False``): what is exchanged between ranks and what a caller accumulates over the slides of a step."""
        return self._bufs

    def load(self, packed: Dict):
        """Copy one packed slide (pinned host or device tensors of the captured shapes) into the static inputs.  A slide
        announced with ``prefetch`` is already in the device staging buffers: it costs one device-to-device copy."""
        if packed is self._staged_for:
            torch.cuda.current_stream().wait_event(self._staged_evt)
            for k, v in self.static.items():
                v.copy_(self._staging[k], non_blocking=True)
            self._consumed_evt.record()
            self._staged_for = None
            return
        for k, v in self.static.items():
            v.copy_(packed[k], non_blocking=True)

    def prefetch(self, packed: Dict):
        """Double buffering of the input path (the job of the reference's pinned-memory DataLoader workers,
        utils/base_trainer.py:283-300): start the host-to-device copy of the NEXT slide on a copy stream, into staging
        buffers, while the current step runs.  The copy waits only for the previous consumer of the staging buffers,
        not for the step in flight; ``load`` of the same ``packed`` object then takes it from there."""
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
            self._staging = {k: torch.empty_like(v) for k, v in self.static.items()}
            self._staged_evt, self._consumed_evt = torch.cuda.Event(), torch.cuda.Event()
            self._consumed_evt.record()
        self._copy_stream.wait_event(self._consumed_evt)
        with torch.cuda.stream(self._copy_stream):
            for k, v in self._staging.items():
                v.copy_(packed[k], non_blocking=True)
            self._staged_evt.record()
        self._staged_for = packed

    def read_back_async(self):
        """Queue the device-to-host copy of this step's (loss, logits) into pinned buffers (a ring of two, so the caller
        may launch the NEXT step before it waits) and return (event, loss_host [1], logits_host): the training loop's
        ``loss.item()`` without stalling the GPU between steps -- the host reads step i while step i + 1 runs."""
        if not hasattr(self, "_rb"):
            mk = lambda t: torch.empty(t.shape, dtype=torch.float32).pin_memory()
            self._rb = [(mk(self.loss.reshape(1)), mk(self.logits), torch.cuda.Event()) for _ in range(2)]
            self._rb_i = 0
        lh, gh, ev = self._rb[self._rb_i]
        self._rb_i ^= 1
        lh.copy_(self.loss.reshape(1), non_blocking=True)
        gh.copy_(self.logits.float(), non_blocking=True)
        ev.record()
        return ev, lh, gh

    def __call__(self, packed: Optional[Dict] = None, reduce: bool = True):
        """``reduce``: all-reduce the flat gradients over the data-parallel ranks after the replay (one slide per rank and
        step).  ``GraphCache`` passes False: ranks step through different numbers of slides and exchange the accumulated
        gradients once."""
        if self._capture_signature() != self._signature:
            # the graph holds pointers to bf16 copies derived from the old frozen weights, or was captured with the
            # other setting of the deterministic switch: capture again
            self._capture()
        if packed is not None:
            self.load(packed)
        self.graph.replay()
        import torch.distributed as dist

        if reduce and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            assert self._bufs is not None, "a step captured with flatten=False cannot exchange its gradients"
            for b in self._bufs:
                dist.all_reduce(b, op=dist.ReduceOp.SUM)
            torch._foreach_div_(self._bufs, float(dist.get_world_size()))
        # ``optimizer.zero_grad()`` (set_to_none, the reference's loop) or ``flat.zero()`` drop ``p.grad``; the replay
        # has rewritten the flat buffer, so every parameter gets its view back and ``optimizer.step()`` sees it
        for p, g in zip(self.flat.params, self._grad_views):
            p.grad = g
        return self.loss, self.logits


class GraphCache:
    """Captured steps for VARIABLE-length slides (pan-cancer training, BASELINE config 5: 2k-40k tiles per slide).

    A CUDA graph is shape-specific and the eager step is host-bound (~3 000 launches from Python: twice the graph's
    time at 10k tiles, worse below), but training visits the same slides every epoch: the cache keeps one captured step
    per token count.  All steps share ONE memory pool and ONE set of static input buffers sized for ``max_tiles`` --
    they are replayed one at a time and their outputs (loss, logits, flat gradients) are consumed before the next
    replay -- so a cached shape costs only its graph object, not its 13-50 GB of activations.  The first visit of a shape
    captures (about the cost of an eager step); every later visit is one graph launch.  ``hits`` / ``misses`` count."""

    def __init__(self, model, projector, flat: FlatGradAllReduce, sizes: Sequence[int], in_chans: int = 1536,
                 max_tiles: int = 40960, max_entries: int = 4096):
        from collections import OrderedDict
        self.model, self.projector, self.flat, self.sizes = model, projector, flat, list(sizes)
        dev = next(model.parameters()).device
        self.pool = torch.cuda.graph_pool_handle()
        self.max_tiles, self.max_entries = max_tiles, max_entries
        self._x = torch.empty((max_tiles, in_chans), device=dev, dtype=torch.float32)
        self._coords = torch.empty((max_tiles, 2), device=dev, dtype=torch.float32)
        self._small: Dict[str, torch.Tensor] = {}
        self.steps: "OrderedDict[int, GraphedStep]" = OrderedDict()
        self.hits = self.misses = 0

    def _static_for(self, packed: Dict) -> Dict:
        L = packed["x"].shape[-2]
        assert L <= self.max_tiles, f"slide of {L} tiles exceeds max_tiles={self.max_tiles}"
        out = {}
        for k, v in packed.items():
            if k == "x":
                out[k] = self._x[:L].view(v.shape)
            elif k == "coords":
                out[k] = self._coords[:L].view(v.shape)
            else:
                if k not in self._small:
                    self._small[k] = torch.empty(v.shape, device=self._x.device, dtype=v.dtype)
                out[k] = self._small[k]
        return out

    def __call__(self, packed: Dict):
        """One slide step (packed host or device tensors, ``pack_host_slide``): (loss, logits); the gradients of THIS
        slide are in ``p.grad`` (views of the captured step's flat buffer, valid until the next call).  No collective
        runs here: a rank's slides of a global step differ in number, the caller accumulates and all-reduces once."""
        L = int(packed["x"].shape[-2])
        step = self.steps.get(L)
        if step is None:
            self.misses += 1
            if len(self.steps) >= self.max_entries:
                self.steps.popitem(last=False)
            self.flat.zero()
            step = GraphedStep(self.model, self.projector, packed, self.sizes, self.flat,
                               warmup=1 if not self.steps else 0, pool=self.pool, static=self._static_for(packed),
                               flatten=True)   # the caller accumulates the slides of a global step: one flat vector
            self.steps[L] = step
            return step(reduce=False)
        self.hits += 1
        self.steps.move_to_end(L)
        return step(packed, reduce=False)
