"""The forward-only inference path on CPU (host logic, kernels replaced by the stand-ins of ``tests/cpu_kernels.py``):
task passes in lockstep through the frozen layers, the batched frozen layer, when each is chosen, and the cache of
captured evaluation forwards (its keys, re-captures and refusals; the graphs themselves need the B200).  The two
batched wrappers (``ops.dilated_attn_fwd_batch``, ``ops.dilated_merge_ln_fwd_batch``) get their stand-ins here, built
on the per-sequence stand-ins."""
import contextlib
import types

import pytest
import torch

from modaltune_b200 import config, ops, synthetic, train_step
from modaltune_b200.longvit_adapter import LongNetGeneAdapter
from tests import cpu_kernels, helpers


@pytest.fixture(scope="module", params=[True, False], ids=["clinical", "gene"])
def model(request):
    return helpers.build_model(helpers.SMALL_GROUPS, clinical=request.param)


def _forward_tasks(model, slide):
    eye = torch.eye(train_step.NUM_TASKS)
    clinical = slide["clinical"] if model._HAS_CLINICAL else None
    return model.forward_tasks(slide["x"], slide["coords"], slide["genes"], clinical, [eye[t] for t in range(3)])


def _attn_fwd_batch(geom, qkv, impl):
    outs = [cpu_kernels.dilated_attn_fwd(geom, qkv[b], impl) for b in range(qkv.shape[0])]
    return torch.cat([o for o, _ in outs]), torch.cat([l for _, l in outs])


def _merge_ln_fwd_batch(geom, o_br, lse_br, gamma, beta, batch, eps=1e-5):
    no, nl = geom.o_elems, geom.lse_elems
    return torch.cat([cpu_kernels.dilated_merge_ln_fwd(geom, o_br[b * no:(b + 1) * no], lse_br[b * nl:(b + 1) * nl],
                                                       gamma, beta, eps)[0] for b in range(batch)])


@contextlib.contextmanager
def _kernels():
    """``cpu_kernels.installed()`` plus the stand-ins of the batched wrappers."""
    saved = (ops.dilated_attn_fwd_batch, ops.dilated_merge_ln_fwd_batch)
    try:
        with cpu_kernels.installed():
            ops.dilated_attn_fwd_batch, ops.dilated_merge_ln_fwd_batch = _attn_fwd_batch, _merge_ln_fwd_batch
            yield
    finally:
        ops.dilated_attn_fwd_batch, ops.dilated_merge_ln_fwd_batch = saved


class _Count:
    def __init__(self, monkeypatch, owner, name):
        self.calls = []
        real = getattr(owner, name)

        def spy(*a, **kw):
            self.calls.append(a)
            return real(*a, **kw)

        monkeypatch.setattr(owner, name, spy)


def test_lockstep_equals_the_per_pass_forward_fp32(model, monkeypatch):
    """The lockstep orchestration (every pass's Injector, ONE call of each frozen layer on the [3, N, 768] stack, every
    pass's Extractors) against three separate passes, in fp32.  Lockstep is forced here: in fp32 mode the layers then run
    their per-sequence loop, so what differs from the per-pass forward is the orchestration alone."""
    slide = synthetic.synthetic_slide(150, seed=41, group_sizes=helpers.SMALL_GROUPS)
    with _kernels(), config.using(mode="fp32"), torch.no_grad():
        per_pass = _forward_tasks(model, slide)
        monkeypatch.setattr(LongNetGeneAdapter, "_lockstep", lambda self, n: n > 1)
        lock = _Count(monkeypatch, LongNetGeneAdapter, "_forward_lockstep")
        layer_in = []
        hooks = [l.register_forward_pre_hook(lambda m, a, kw: layer_in.append(a[0].shape[0]), with_kwargs=True)
                 for l in model.encoder.layers]
        try:
            lockstep = _forward_tasks(model, slide)
        finally:
            for h in hooks:
                h.remove()
    assert len(lock.calls) == 1
    assert layer_in == [3] * len(model.encoder.layers)        # each frozen layer once, on the stack of the passes
    assert per_pass.shape == lockstep.shape == (3, 256)
    assert helpers.relerr(lockstep, per_pass) < 1e-6


def test_lockstep_with_batched_layers_bf16(model, monkeypatch):
    """bf16 mode with the tcgen05-GEMM path (stand-ins): forward_tasks without autograd runs lockstep, and every frozen
    layer takes the batched forward; its logits agree with the grad-enabled per-pass forward of the same slide (fp32 CPU
    stand-ins round to bf16 at the same places on both sides; the B200 test compares bitwise)."""
    slide = synthetic.synthetic_slide(200, seed=42, group_sizes=helpers.SMALL_GROUPS)
    with _kernels(), config.using(mode="bf16", gemm="sm100"):
        per_pass = _forward_tasks(model, slide).detach()
        batched = _Count(monkeypatch, ops, "encoder_layer_forward_batch")
        with torch.no_grad():
            lockstep = _forward_tasks(model, slide)
    assert len(batched.calls) == len(model.encoder.layers)
    assert all(c[3] == 3 for c in batched.calls)
    assert helpers.relerr(lockstep, per_pass) < 1e-2


@pytest.mark.parametrize("n", [200, 256, 129])
def test_batched_layer_equals_per_sequence_calls(n):
    """The batched frozen layer (qkv padded per sequence, attention and merge per sequence block, everything else on the
    stacked rows) against one call per sequence, with different inputs per sequence (bf16 mode, stand-ins)."""
    model = helpers.build_model(helpers.SMALL_GROUPS)
    layer = model.encoder.layers[0]
    torch.manual_seed(n)
    x = torch.randn(3, n, 768)
    with _kernels(), config.using(mode="bf16", gemm="sm100"), torch.no_grad():
        assert layer.runs_batched(x)
        y, _ = layer(x)
        want = torch.cat([layer(x[b:b + 1])[0] for b in range(3)], 0)
    assert y.shape == (3, n, 768)
    for b in range(3):
        assert helpers.relerr(y[b], want[b]) < 1e-2, b


def test_fallback_conditions_select_the_old_paths(model):
    """Lockstep passes and the batched layer only without autograd, in eval mode, in bf16 mode with the tcgen05 GEMMs,
    and (lockstep) with no hooked attention module; every other case keeps the per-pass forward and the layer loop."""
    layer = model.encoder.layers[0]
    x = torch.zeros(3, 16, 768)
    xg = x.clone().requires_grad_(True)
    with config.using(mode="bf16", gemm="sm100"):
        with torch.no_grad():
            assert model._lockstep(3) and layer.runs_batched(x)
            assert not model._lockstep(1) and not layer.runs_batched(x[:1])
            h = model.interactions[0].extractor.attn.multihead_attn.register_forward_hook(lambda *a: None)
            assert not model._lockstep(3)
            h.remove()
            assert model._lockstep(3)
            model.train()
            try:
                assert not model._lockstep(3) and not layer.runs_batched(x)
            finally:
                model.eval()
        assert not model._lockstep(3)                     # grad enabled: autograd would record the passes
        assert not layer.runs_batched(xg)
        assert layer.runs_batched(x)                      # grad enabled, but the input does not require it
    with torch.no_grad():
        with config.using(mode="fp32"):
            assert not model._lockstep(3) and not layer.runs_batched(x)
        with config.using(mode="bf16", gemm="cublas"):
            assert not model._lockstep(3) and not layer.runs_batched(x)


def test_eval_cache_keys_recaptures_and_refusals(monkeypatch):
    """GraphedForwardCache: one captured forward per token count, replays for revisited counts; a re-capture after a
    load_state_dict and after a train / eval switch; a hooked attention module is refused at capture and at replay; no
    gradient is touched.  The capture itself is replaced by a recorder (CUDA graphs need the device)."""
    model = helpers.build_model(helpers.SMALL_GROUPS)
    captures = []

    def fake_capture(self):
        self._check_no_hooks()
        captures.append(int(self.static["x"].shape[-2]))
        self.graph = types.SimpleNamespace(replay=lambda: None)
        self.logits = self.static["x"]
        self._signature = self._capture_signature()

    monkeypatch.setattr(train_step.GraphedForward, "_capture", fake_capture)
    monkeypatch.setattr(torch.cuda, "graph_pool_handle", lambda: None)
    slides = {n: train_step.pack_host_slide(synthetic.synthetic_slide(n, seed=n, group_sizes=helpers.SMALL_GROUPS),
                                            pin=False) for n in (40, 64, 90)}
    sizes = slides[40][1]
    cache = train_step.GraphedForwardCache(model, sizes, max_tiles=128)
    for n in (40, 64, 40, 90, 64):
        out = cache(slides[n][0])
        assert torch.equal(out, slides[n][0]["x"])       # the static inputs hold this slide when the graph replays
    assert (cache.hits, cache.misses) == (2, 3) and captures == [40, 64, 90]
    assert list(cache.steps) == [40, 90, 64]             # least recently used first
    model.load_state_dict(model.state_dict())            # frozen weights rewritten in place: derived copies are stale
    cache(slides[90][0])
    assert captures[-1] == 90 and len(captures) == 4
    cache(slides[90][0])
    assert len(captures) == 4
    model.train()
    try:
        cache(slides[90][0])
        assert len(captures) == 5
    finally:
        model.eval()
    cache(slides[90][0])
    assert len(captures) == 6
    h = model.interactions[2].extra_extractors[0].attn.multihead_attn.register_forward_hook(lambda *a: None)
    with pytest.raises(RuntimeError, match=r"interactions\.2\.extra_extractors\.0\.attn\.multihead_attn"):
        cache(slides[64][0])
    new = train_step.pack_host_slide(synthetic.synthetic_slide(33, seed=3, group_sizes=helpers.SMALL_GROUPS), pin=False)
    with pytest.raises(RuntimeError, match="forward hooks"):
        cache(new[0])                                    # refused at capture too
    h.remove()
    assert cache(slides[64][0]) is not None
    assert all(p.grad is None for p in model.parameters())
    with pytest.raises(AssertionError, match="max_tiles"):
        cache(train_step.pack_host_slide(synthetic.synthetic_slide(129, seed=1, group_sizes=helpers.SMALL_GROUPS),
                                         pin=False)[0])
