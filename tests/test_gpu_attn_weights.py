"""Attention maps of the Modal Adapter on the B200: the ``mt_cross_attn_probs`` kernel (both impls) against float64
references, the maps forward hooks receive from the bf16 model against the base class's float64 forward, and graph
capture with hooks."""
import copy
import math

import pytest
import torch
import torch.nn as nn

from modaltune_b200 import _lib, adapter_modules, config, ops, synthetic, train_step
from tests import helpers

pytestmark = pytest.mark.gpu
DEV = "cuda"
H, E = 12, 192
LOG2E = 1.4426950408889634
# largest deviations seen by the tests of this file, printed at the end of the session (pytest -s) for the record
MEASURED = {}


def _note(key, value):
    MEASURED[key] = max(MEASURED.get(key, 0.0), float(value))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k, v in sorted(MEASURED.items()):
        print(f"measured {k}: {v:.3e}")


def _tf32(x):
    """cvt.rna.tf32.f32: round the fp32 mantissa to 10 bits, ties away from zero."""
    b = x.float().contiguous().view(torch.int32)
    return ((b + 0x1000) & -0x2000).view(torch.float32)


def _heads(t):
    return t.reshape(t.shape[0], H, -1).transpose(0, 1)


def _probs(q, k, lse, impl, pad):
    """mt_cross_attn_probs into a NaN-filled [lq, lk + pad] buffer (row stride lk + pad)."""
    lq, lk = q.shape[0], k.shape[0]
    buf = torch.full((lq, lk + pad), float("nan"), device=DEV)
    rc = _lib.load().mt_cross_attn_probs(ops._ptr(q), q.stride(0), ops._ptr(k), k.stride(0), _lib.MT_F32, ops._p(lse),
                                         ops._p(buf), buf.stride(0), lq, lk, H, E // H, impl, ops._stream())
    assert rc == 0, _lib.last_error()
    return buf


def _tight_reference(q, k, lse, impl):
    """float64 from the operands the kernel multiplies and the forward's lse: impl 1 = TF32-rounded q * log2(e)/4 and
    TF32-rounded k, scores in the log2 domain against lse * log2(e) (both products in fp32, as on the device)."""
    if impl == 1:
        c = torch.tensor(0.25, dtype=torch.float32) * torch.tensor(LOG2E, dtype=torch.float32)
        s = _heads(_tf32(q * c).double()) @ _heads(_tf32(k).double()).transpose(1, 2)
        L = (lse * torch.tensor(LOG2E, dtype=torch.float32, device=DEV)).double().t()[..., None]
        return torch.exp2(s - L).mean(0)
    s = _heads((q * 0.25).double()) @ _heads(k.double()).transpose(1, 2)
    return torch.exp(s - lse.double().t()[..., None]).mean(0)


def _exact(q, k):
    """The head-averaged softmax(q k^T / 4) in float64 on the unrounded inputs (nn.MultiheadAttention's weights)."""
    s = _heads(q.double()) @ _heads(k.double()).transpose(1, 2) / 4.0
    return torch.softmax(s, -1).mean(0)


def assert_maps_close(got, want, rel):
    """|got - want| <= rel * (row maximum of want), element by element; returns the largest ratio."""
    assert got.shape == want.shape
    err = (got.double() - want).abs() / want.amax(-1, keepdim=True).clamp_min(1e-300)
    worst = float(err.max())
    assert worst <= rel, worst
    return worst


SHAPES = [(10001, 66), (66, 10000), (66, 32768), (66, 66), (1, 17), (17, 1), (73, 1025), (1025, 73), (17, 73)]


@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("layout", ["kv384", "shared1152"])
@pytest.mark.parametrize("lq,lk", SHAPES)
def test_probs_kernel_against_float64(lq, lk, layout, impl):
    g = torch.Generator(device=DEV).manual_seed(lq * 131 + lk)
    q = torch.randn(lq, E, device=DEV, generator=g)
    width, col0, pad = (384, 0, 0) if layout == "kv384" else (1152, 384, 2)   # the 2nd extractor's slice of the shared buffer
    kv = torch.randn(lk, width, device=DEV, generator=g)
    k, v = kv[:, col0:col0 + E], kv[:, col0 + E:col0 + 2 * E]
    _, lse = ops.cross_attn_fwd(q, k, v, H, impl=impl)
    buf = _probs(q, k, lse, impl, pad)
    p = buf[:, :lk]
    assert not bool(torch.isnan(p).any()), "unwritten output elements"
    assert bool(torch.isnan(buf[:, lk:]).all()), "written outside [lq, lk]"
    tight = _tight_reference(q, k, lse, impl)
    bound = 1e-6 + 1e-5 * tight.abs()
    excess = float(((p.double() - tight).abs() - bound).max())
    _note(f"impl{impl} tight |P - ref| / (1e-6 + 1e-5 |ref|)", float(((p.double() - tight).abs() / bound).max()))
    assert excess <= 0, excess
    _note(f"impl{impl} loose (row-max units)", assert_maps_close(p, _exact(q, k), 5e-3 if impl == 1 else 1e-5))
    rows = p.double().sum(-1)
    _note(f"impl{impl} |row sum - 1|", (rows - 1).abs().max())
    assert float((rows - 1).abs().max()) < 1e-5
    again = _probs(q, k, lse, impl, pad)
    assert torch.equal(again.view(torch.int32), buf.view(torch.int32))        # bitwise repeatable (NaN pad included)
    if layout == "kv384":
        assert torch.equal(ops.cross_attn_probs(q, k, lse, H, impl=impl), p)   # the wrapper runs the same launch


def test_map_assertion_rejects_wrong_references():
    """Negative control: the helper used above fails against a transposed map and against one head instead of the
    average."""
    g = torch.Generator(device=DEV).manual_seed(5)
    q = torch.randn(66, E, device=DEV, generator=g)
    kv = torch.randn(66, 384, device=DEV, generator=g)
    k, v = kv[:, :E], kv[:, E:]
    _, lse = ops.cross_attn_fwd(q, k, v, H, impl=1)
    p = ops.cross_attn_probs(q, k, lse, H, impl=1)
    want = _exact(q, k)
    assert_maps_close(p, want, 5e-3)
    with pytest.raises(AssertionError):
        assert_maps_close(p, want.t().contiguous(), 5e-3)
    one_head = torch.softmax(_heads(q.double())[0] @ _heads(k.double())[0].t() / 4.0, -1)
    with pytest.raises(AssertionError):
        assert_maps_close(p, one_head, 5e-3)


def _mhas(model):
    return [(n, m) for n, m in model.named_modules() if isinstance(m, nn.MultiheadAttention)]


def _step(model, proj, slide):
    for p in model.parameters():
        p.grad = None
    _, logits = train_step.forward_backward(model, proj, slide)
    torch.cuda.synchronize()
    return logits.clone(), torch.cat([p.grad.reshape(-1).double() for p in model.parameters()
                                      if p.requires_grad and p.grad is not None])


@pytest.mark.parametrize("pathways", ["toy10", "full331"])
def test_bf16_model_maps_match_the_reference_forward(pathways):
    """bf16 mode, 10k tiles, 3 task passes on their streams: every map a hook receives matches the base class's float64
    forward on the inputs the hook saw (row-max bound of the TF32 kernel), and the step with hooks equals the step
    without them (the bars of the host restructurings, DESIGN.md §2)."""
    groups = helpers.SMALL_GROUPS if pathways == "toy10" else None
    model = helpers.build_model(groups, device=DEV)
    proj = helpers.build_projector(0, DEV)
    slide = train_step.slide_to_device(synthetic.synthetic_slide(10000, seed=41, group_sizes=groups), DEV)
    seen, handles = [], []
    for name, m in _mhas(model):
        def hook(mod, args, kwargs, out, name=name, m=m):
            k = kwargs["key"]
            seen.append((name, m, kwargs["query"].detach().clone(), k.detach().clone(),
                         None if kwargs["value"] is k else kwargs["value"].detach().clone(), out[1]))
        handles.append(m.register_forward_hook(hook, with_kwargs=True))
    with config.using(mode="bf16"):
        try:
            hooked = _step(model, proj, slide)
        finally:
            for h in handles:
                h.remove()
        plain = _step(model, proj, slide)
    assert len(seen) == len(_mhas(model)) * train_step.NUM_TASKS
    for name, m, q, k, v, w in seen:
        m64 = copy.deepcopy(m).double()
        with torch.no_grad():
            k64 = k.double()
            _, ref = nn.MultiheadAttention.forward(m64, q.double(), k64, k64 if v is None else v.double())
        assert w.dtype == torch.float32 and w.shape == ref.shape
        _note(f"model {pathways} map (row-max units)", assert_maps_close(w[0], ref[0], 5e-3))
    rel = helpers.relerr(hooked[0], plain[0])
    a, b = hooked[1], plain[1]
    cos = float(a @ b / (a.norm() * b.norm()))
    _note(f"model {pathways} logits relerr", rel)
    _note(f"model {pathways} 1 - grad cosine", 1 - cos)
    assert rel < 5e-3
    assert cos > 0.9999


def test_graph_capture_refuses_hooks_and_captures_after_remove():
    model = helpers.build_model(helpers.SMALL_GROUPS, device=DEV)
    proj = helpers.build_projector(0, DEV)
    flat = train_step.FlatGradAllReduce([p for p in model.parameters() if p.requires_grad])
    packed, sizes, _ = train_step.pack_host_slide(synthetic.synthetic_slide(700, seed=42, group_sizes=helpers.SMALL_GROUPS))
    mha = model.prompt_selfattention[1].self_attn
    h = mha.register_forward_pre_hook(lambda *a: None)
    with config.using(mode="bf16"):
        with pytest.raises(RuntimeError, match=r"prompt_selfattention\.1\.self_attn"):
            train_step.GraphedStep(model, proj, packed, sizes, flat)
        h.remove()
        step = train_step.GraphedStep(model, proj, packed, sizes, flat)
        loss, _ = step(packed)
        assert math.isfinite(float(loss))
        h = mha.register_forward_hook(lambda *a: None)   # registered after capture: the replay would skip it
        with pytest.raises(RuntimeError, match="forward hooks"):
            step(packed)
        h.remove()
    assert adapter_modules.hooked_attention(model.named_modules()) == []
