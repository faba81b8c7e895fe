"""Attention maps of the Modal Adapter through forward hooks (host logic, CPU).

The adapter layers call their attention arithmetic directly and go through ``adapter_modules.MultiheadAttention`` (an
``nn.MultiheadAttention``) only when that module has a forward hook or pre-hook; a hook then receives the reference's
``need_weights=True`` output.  The kernels are replaced by the torch stand-ins of ``tests/cpu_kernels.py``; the stand-in
of ``ops.cross_attn_probs`` lives in the ``probs`` fixture below.
"""
import copy
import math

import pytest
import torch
import torch.nn as nn

from modaltune_b200 import adapter_modules, config, ops, synthetic, train_step
from modaltune_b200.adapter_modules import MultiheadAttention
from tests import cpu_kernels, helpers


def _heads(t, heads):
    return t.reshape(t.shape[0], heads, -1).transpose(0, 1)


def _fwd_standin(q, k, v, heads, impl=None):
    """cross_attn_fwd in the operands' own precision (float64 for the module-level check)."""
    qh, kh, vh = _heads(q, heads), _heads(k, heads), _heads(v, heads)
    s = qh @ kh.transpose(1, 2) / math.sqrt(qh.shape[-1])
    lse = torch.logsumexp(s, -1)
    return (torch.exp(s - lse[..., None]) @ vh).transpose(0, 1).reshape(q.shape), lse.t().contiguous()


def _probs_standin(q, k, lse, heads, impl=None):
    """mt_cross_attn_probs: (1/H) sum_h exp(q k^T / sqrt(d) - lse), in float64, returned as fp32 (or float64 operands'
    precision)."""
    qh, kh = _heads(q.double(), heads), _heads(k.double(), heads)
    s = qh @ kh.transpose(1, 2) / math.sqrt(qh.shape[-1])
    p = torch.exp(s - lse.double().t()[..., None]).mean(0)
    return p.to(torch.promote_types(q.dtype, torch.float32))


@pytest.fixture
def probs(monkeypatch):
    monkeypatch.setattr(ops, "cross_attn_probs", _probs_standin)


@pytest.fixture(scope="module", params=[True, False], ids=["clinical", "gene"])
def model(request):
    return helpers.build_model(helpers.SMALL_GROUPS, clinical=request.param)


def _mhas(model):
    return [(n, m) for n, m in model.named_modules() if isinstance(m, nn.MultiheadAttention)]


def _step(model, slide, proj):
    for p in model.parameters():
        p.grad = None
    loss, logits = train_step.forward_backward(model, proj, slide)
    return logits.clone(), {n: p.grad.clone() for n, p in model.named_parameters() if p.requires_grad and p.grad is not None}


def _capture_hooks(model):
    seen, handles = {}, []
    for name, m in _mhas(model):
        def hook(mod, args, kwargs, out, name=name):
            assert args == ()
            q, k, v = kwargs["query"], kwargs["key"], kwargs["value"]
            seen.setdefault(name, []).append((q.detach().clone(), k.detach().clone(), v.detach().clone(), k is v,
                                              out[0].detach().clone(), out[1]))
        handles.append(m.register_forward_hook(hook, with_kwargs=True))
    return seen, handles


def _base_mha(m, q, k, v, same):
    """nn.MultiheadAttention.forward of the base class in float64 on the captured inputs."""
    m64 = copy.deepcopy(m).double()
    k64 = k.double()
    with torch.no_grad():
        return nn.MultiheadAttention.forward(m64, q.double(), k64, k64 if same else v.double(), need_weights=True)


def test_hooks_receive_the_reference_weights_and_change_nothing(model, probs):
    """Hooks on every attention module of the adapter: each fires once per task pass, receives (attn_output, weights)
    equal to the base class's float64 forward on the inputs it was called with, and the step (logits, gradients) is the
    step without hooks."""
    slide = synthetic.synthetic_slide(120, seed=31, group_sizes=helpers.SMALL_GROUPS)
    proj = helpers.build_projector(0)
    mhas = _mhas(model)
    assert len(mhas) == 10 and all(isinstance(m, MultiheadAttention) for _, m in mhas)
    with cpu_kernels.installed(), config.using(mode="fp32"):
        plain = _step(model, slide, proj)
        seen, handles = _capture_hooks(model)
        try:
            hooked = _step(model, slide, proj)
        finally:
            for h in handles:
                h.remove()
    assert sorted(seen) == sorted(n for n, _ in mhas)
    worst_w = worst_o = 0.0
    for name, calls in seen.items():
        assert len(calls) == train_step.NUM_TASKS, name
        for q, k, v, same, out, w in calls:
            assert w.dtype == torch.float32 and not w.requires_grad
            assert w.shape == (1, q.shape[1], k.shape[1]) and out.shape == q.shape
            ref_o, ref_w = _base_mha(dict(mhas)[name], q, k, v, same)
            worst_w = max(worst_w, float((w.double() - ref_w).abs().max()))
            worst_o = max(worst_o, float((out.double() - ref_o).abs().max() / ref_o.abs().max()))
            torch.testing.assert_close(w.double().sum(-1), torch.ones_like(ref_w.sum(-1)), rtol=0, atol=1e-5)
    # fp32 projections and scores against float64 ones: the weights agree to fp32 rounding (7e-8 measured)
    assert worst_w < 1e-6, worst_w
    assert worst_o < 1e-5, worst_o
    assert helpers.relerr(hooked[0], plain[0]) < 2e-4
    assert set(hooked[1]) == set(plain[1])
    gmax = max(float(g.abs().max()) for g in plain[1].values())
    for n, g in plain[1].items():
        if float(g.abs().max()) < 1e-6 * gmax:
            continue
        assert helpers.relerr(hooked[1][n], g) < 2e-4, n


def test_module_forward_is_the_base_class_forward_in_float64(monkeypatch, probs):
    """The subclass's own arithmetic (projections, packed k | v when key is value, head average) against
    nn.MultiheadAttention.forward, both in float64: agreement to float64 rounding."""
    monkeypatch.setattr(ops, "cross_attn_fwd", _fwd_standin)
    torch.manual_seed(3)
    m = MultiheadAttention(192, 12, batch_first=True, kdim=768, vdim=768).double()
    nn.init.normal_(m.in_proj_bias, std=0.1)
    nn.init.normal_(m.out_proj.bias, std=0.1)
    q = torch.randn(1, 17, 192, dtype=torch.float64)
    k = torch.randn(1, 73, 768, dtype=torch.float64)
    v = torch.randn(1, 73, 768, dtype=torch.float64)
    with config.using(mode="fp32"):
        for key, value in ((k, k), (k, v)):
            out, w = m(q, key, value)
            ref_o, ref_w = nn.MultiheadAttention.forward(m, q, key, value)
            assert float((w - ref_w).abs().max()) < 1e-10
            assert float((out - ref_o).abs().max()) < 1e-10
            out2, none = m(q, key, value, need_weights=False)
            assert none is None and torch.equal(out2, out)


class _Spy:
    def __init__(self, monkeypatch, mod, name):
        self.calls = 0
        real = getattr(mod, name)

        def spy(*a, **kw):
            self.calls += 1
            return real(*a, **kw)

        monkeypatch.setattr(mod, name, spy)


def _forward_counts(model, slide, monkeypatch):
    inj, kv = _Spy(monkeypatch, ops, "injector"), _Spy(monkeypatch, ops, "shared_kv_project")
    mha = _Spy(monkeypatch, MultiheadAttention, "forward")
    with torch.no_grad():
        train_step.multitask_forward(model, slide)
    return inj.calls, kv.calls, mha.calls


def test_fused_paths_run_unless_a_module_is_hooked(model, probs, monkeypatch):
    """Without hooks the fused Injector and the shared k | v projection of the last block run and no attention module is
    called; a hook on one extractor of the last block sends that block to the per-extractor path, a hook on an injector
    takes it off the fused node; removing the hooks restores both."""
    slide = synthetic.synthetic_slide(64, seed=32, group_sizes=helpers.SMALL_GROUPS)
    last = model.interactions[-1]
    n_blocks, tasks = len(model.interactions), train_step.NUM_TASKS
    with cpu_kernels.installed(), config.using(mode="fp32"):
        assert _forward_counts(model, slide, monkeypatch) == (n_blocks * tasks, tasks, 0)
        h1 = last.extra_extractors[0].attn.multihead_attn.register_forward_hook(lambda *a: None)
        assert _forward_counts(model, slide, monkeypatch) == (n_blocks * tasks, 0, tasks)
        h2 = model.interactions[0].injector.attn.multihead_attn.register_forward_pre_hook(lambda *a: None)
        assert _forward_counts(model, slide, monkeypatch) == ((n_blocks - 1) * tasks, 0, 2 * tasks)
        h1.remove()
        h2.remove()
        assert _forward_counts(model, slide, monkeypatch) == (n_blocks * tasks, tasks, 0)


def test_a_hook_that_replaces_the_output_replaces_it(model, probs):
    """torch's semantics: what a forward hook returns is the module's output.  Zeroing the attention output of one
    extractor through a hook gives the logits of the same model with that extractor's out_proj zeroed."""
    slide = synthetic.synthetic_slide(64, seed=33, group_sizes=helpers.SMALL_GROUPS)
    mha = model.interactions[-1].extra_extractors[1].attn.multihead_attn
    with cpu_kernels.installed(), config.using(mode="fp32"), torch.no_grad():
        base = train_step.multitask_forward(model, slide)
        h = mha.register_forward_hook(lambda m, a, out: (torch.zeros_like(out[0]), out[1]))
        try:
            replaced = train_step.multitask_forward(model, slide)
        finally:
            h.remove()
        saved = [p.clone() for p in (mha.out_proj.weight, mha.out_proj.bias)]
        try:
            mha.out_proj.weight.zero_()
            mha.out_proj.bias.zero_()
            want = train_step.multitask_forward(model, slide)
        finally:
            mha.out_proj.weight.copy_(saved[0])
            mha.out_proj.bias.copy_(saved[1])
    assert helpers.relerr(replaced, base) > 1e-3
    assert helpers.relerr(replaced, want) < 1e-5


@pytest.mark.parametrize("kwargs", [{"attn_mask": torch.zeros(5, 7, dtype=torch.bool)},
                                    {"key_padding_mask": torch.zeros(1, 7, dtype=torch.bool)},
                                    {"average_attn_weights": False}, {"is_causal": True}],
                         ids=["attn_mask", "key_padding_mask", "per_head", "is_causal"])
def test_masks_and_per_head_weights_raise(kwargs):
    m = MultiheadAttention(192, 12, batch_first=True, kdim=768, vdim=768)
    with pytest.raises(NotImplementedError):
        m(torch.randn(1, 5, 192), torch.randn(1, 7, 768), torch.randn(1, 7, 768), **kwargs)


def test_graph_capture_refuses_a_hooked_model():
    """A hook runs on the host: it would run once at capture and never on replay, so capture raises and names the module.
    (The check runs before anything touches a device.)"""
    model = helpers.build_model(helpers.SMALL_GROUPS)
    slide = synthetic.synthetic_slide(32, seed=34, group_sizes=helpers.SMALL_GROUPS)
    packed, sizes, _ = train_step.pack_host_slide(slide, pin=False)
    h = model.interactions[1].extractor.attn.multihead_attn.register_forward_hook(lambda *a: None)
    flat = train_step.FlatGradAllReduce([p for p in model.parameters() if p.requires_grad])
    with pytest.raises(RuntimeError, match=r"interactions\.1\.extractor\.attn\.multihead_attn"):
        train_step.GraphedStep(model, helpers.build_projector(0), packed, sizes, flat)
    h.remove()
    assert adapter_modules.hooked_attention(model.named_modules()) == []
