"""The forward-only inference path on the B200: batched dilated attention, the forward-only fc1 epilogue, the batched frozen
layer, task passes in lockstep and the captured evaluation forward.  Every comparison with the per-sequence / per-pass
path is bitwise (torch.equal): each kernel of the bf16 forward computes a row or work item the same way whatever the
batch."""
import os

import pytest
import torch

from modaltune_b200 import _lib, config, ops, synthetic, train_step
from modaltune_b200.slide_encoder import DILATED_RATIO, LongNetViT, optimal_segment_lengths
from tests import dilated_ref64 as R
from tests import helpers
from tests.test_gpu_dilated_sm100_ref64 import _qkv, check_fwd

pytestmark = pytest.mark.gpu
DEV = "cuda"
B = 3


def _geom(n):
    return ops.Geometry.get(n, optimal_segment_lengths(), DILATED_RATIO)


def _fwd_batch(geom, qkv, impl):
    """mt_dilated_attn_fwd_batch into NaN-filled outputs: every element must be written."""
    nb = qkv.shape[0]
    o = torch.full((nb * geom.o_elems,), float("nan"), device=DEV, dtype=qkv.dtype)
    lse = torch.full((nb * geom.lse_elems,), float("nan"), device=DEV, dtype=torch.float32)
    rc = _lib.load().mt_dilated_attn_fwd_batch(geom.ref(), ops._p(qkv), qkv.stride(1), geom.n_alloc, nb, ops._dt(qkv),
                                               ops._p(o), ops._p(lse), impl, ops._stream())
    assert rc == 0, _lib.last_error()
    return o, lse


def _fwd_one(geom, qkv, impl):
    o = torch.full((geom.o_elems,), float("nan"), device=DEV, dtype=qkv.dtype)
    lse = torch.full((geom.lse_elems,), float("nan"), device=DEV, dtype=torch.float32)
    rc = _lib.load().mt_dilated_attn_fwd(geom.ref(), ops._p(qkv), qkv.stride(0), geom.n_alloc, ops._dt(qkv), ops._p(o),
                                         ops._p(lse), impl, ops._stream())
    assert rc == 0, _lib.last_error()
    return o, lse


# 1025: one token past a multiple of 128, so the last 1024-token segment holds a single real position
@pytest.mark.parametrize("n", [1025, 1200, 5793, 10001, 32769])
@pytest.mark.parametrize("impl,dtype", [(3, torch.bfloat16), (0, torch.float32)], ids=["impl3-bf16", "simt-fp32"])
def test_attention_batch_equals_single_calls(n, impl, dtype):
    """B = 3 sequences with different random q / k / v in one launch against three single launches: all of o_br and
    lse_br bitwise.  A read across a sequence boundary (the zero fill of the last segments) would show."""
    geom = _geom(n)
    qkv = torch.stack([_qkv(geom, "randn", 100 * n + b) for b in range(B)]).to(dtype).contiguous()
    o, lse = _fwd_batch(geom, qkv, impl)
    for b in range(B):
        o1, lse1 = _fwd_one(geom, qkv[b], impl)
        assert bool(torch.isfinite(o1.float()).all())
        assert torch.equal(o[b * geom.o_elems:(b + 1) * geom.o_elems], o1), (n, impl, b)
        assert torch.equal(lse[b * geom.lse_elems:(b + 1) * geom.lse_elems], lse1), (n, impl, b)


def test_attention_batch_impl3_against_float64():
    """The batched 48-key kernel against the float64 reference of every sequence, within the per-element bound of
    tests/test_gpu_dilated_sm100_ref64.py."""
    geom = _geom(5793)
    regimes = ("randn", "flat", "rising")
    qkv = torch.stack([_qkv(geom, r, 7 + b) for b, r in enumerate(regimes)]).contiguous()
    o, lse = _fwd_batch(geom, qkv, 3)
    torch.cuda.synchronize()
    for b, r in enumerate(regimes):
        ref = R.fwd_ref64(geom, qkv[b])
        check_fwd(o[b * geom.o_elems:(b + 1) * geom.o_elems], lse[b * geom.lse_elems:(b + 1) * geom.lse_elems], ref,
                  f"batched impl 3, sequence {b} {r}")


def test_batch_rejected_by_impl1():
    geom = _geom(1200)
    qkv = torch.zeros(2, geom.n_alloc, 2304, device=DEV, dtype=torch.bfloat16)
    o = torch.empty(2 * geom.o_elems, device=DEV, dtype=torch.bfloat16)
    lse = torch.empty(2 * geom.lse_elems, device=DEV)
    rc = _lib.load().mt_dilated_attn_fwd_batch(geom.ref(), ops._p(qkv), 2304, geom.n_alloc, 2, _lib.MT_BF16, ops._p(o),
                                               ops._p(lse), 1, ops._stream())
    assert rc != 0 and "batch" in _lib.last_error()


def test_forward_only_fc1_epilogue():
    """MT_EPI_GELU_STATS with neither h nor gelu'(h): u and the slab statistics equal the training epilogue's (with
    gelu'(h), and with h)."""
    torch.manual_seed(5)
    M = 3 * 1201
    a = (torch.randn(M, 768, device=DEV) * 0.5).to(torch.bfloat16)
    w = (torch.randn(3072, 768, device=DEV) * 0.03).to(torch.bfloat16)
    bias = torch.randn(3072, device=DEV) * 0.1
    outs = {}
    for kind in ("aux", "h", "none"):
        u = torch.empty(M, 3072, device=DEV, dtype=torch.bfloat16)
        stats = torch.empty(M, 24, 2, device=DEV)
        aux = torch.empty(M, 3072, device=DEV, dtype=torch.bfloat16) if kind == "aux" else None
        ops.linear_sm100(a, w, mode=_lib.MT_EPI_GELU_STATS, bias=bias, want_f32=kind == "h", out_bf16=u, stats=stats,
                         out_aux=aux)
        outs[kind] = (u, stats)
    for kind in ("aux", "h"):
        assert torch.equal(outs["none"][0], outs[kind][0]) and torch.equal(outs["none"][1], outs[kind][1]), kind


@pytest.fixture(scope="module")
def layer():
    m = helpers.build_model(helpers.SMALL_GROUPS, device=DEV)
    return m.encoder.layers[5]


@pytest.mark.parametrize("n", [10001, 32769])
def test_batched_layer_equals_per_sequence_calls(layer, n):
    torch.manual_seed(n)
    x = torch.randn(B, n, 768, device=DEV)
    with config.using(mode="bf16"), torch.no_grad():
        assert layer.runs_batched(x)
        y, _ = layer(x)
        for b in range(B):
            yb, _ = layer(x[b:b + 1])
            assert torch.equal(y[b], yb[0]), (n, b)


def test_longnetvit_batch_of_two_slides():
    """Prov-GigaPath's standard use, ``LongNetViT.forward(tile_embeds, coords, all_layer_embed=True)`` on a batch of two
    slides, against one call per slide: every layer's embedding bitwise."""
    torch.manual_seed(11)
    vit = LongNetViT(in_chans=1536, embed_dim=768, depth=12, mlp_ratio=4.0).to(DEV).eval()
    for p in vit.parameters():
        p.requires_grad_(False)
    L = 2000
    x = torch.randn(2, L, 1536, device=DEV)
    coords = torch.randint(0, 200 * 256, (2, L, 2), device=DEV).float()
    with config.using(mode="bf16"), torch.no_grad():
        both = vit(x, coords, all_layer_embed=True)
        for b in range(2):
            one = vit(x[b:b + 1], coords[b:b + 1], all_layer_embed=True)
            assert len(one) == len(both) == 13
            for k, (u, v) in enumerate(zip(both, one)):
                assert torch.equal(u[b], v[0]), (b, k)


def _tasks(model, slide):
    return train_step.multitask_forward(model, slide)


@pytest.mark.parametrize("clinical", [True, False], ids=["clinical", "gene"])
def test_no_grad_forward_tasks_331_pathways(clinical, monkeypatch):
    """331 pathways, 10 000 tiles: the no-grad forward_tasks (passes in lockstep, batched layers) against the
    grad-enabled forward_tasks of the same model and slide, bitwise; and against the reference's logits of the fixture
    slide within the bf16 bar of tests/test_gpu_model.py."""
    m = helpers.build_model(None, clinical=clinical, device=DEV)
    slide = train_step.slide_to_device(synthetic.synthetic_slide(10000, seed=77), DEV)
    lock = []
    real = type(m)._forward_lockstep
    monkeypatch.setattr(type(m), "_forward_lockstep", lambda *a: lock.append(1) or real(*a))
    with config.using(mode="bf16"):
        with torch.no_grad():
            fast = _tasks(m, slide)
        assert len(lock) == 1
        slow = _tasks(m, slide)
        assert len(lock) == 1
    assert torch.equal(fast, slow.detach())
    if clinical:
        gold = torch.load(os.path.join(helpers.GOLDEN, "training_step_331.pt"))
        fix = train_step.slide_to_device(synthetic.synthetic_slide(gold["L"], seed=gold["seed"]), DEV)
        with config.using(mode="bf16"), torch.no_grad():
            logits = _tasks(m, fix)
        assert len(lock) == 2
        assert helpers.relerr(logits.float().cpu(), gold["logits"]) < 2e-2


def test_graphed_evaluation_equals_eager():
    """GraphedForwardCache against eager no-grad forward_tasks: three token counts, revisited in another order with new
    slides; after a load_state_dict that changes a frozen weight it re-captures and matches the eager forward again."""
    m = helpers.build_model(helpers.SMALL_GROUPS, device=DEV)
    tiles = (700, 333, 1201)
    packs = {n: [train_step.pack_host_slide(synthetic.synthetic_slide(n, seed=s + n, group_sizes=helpers.SMALL_GROUPS))
                 for s in (1, 2)] for n in tiles}
    sizes = packs[700][0][1]

    def eager(packed):
        slide = train_step.unpack_slide({k: v.to(DEV) for k, v in packed.items()}, sizes)
        with torch.no_grad():
            return train_step.multitask_forward(m, slide)

    with config.using(mode="bf16"):
        cache = train_step.GraphedForwardCache(m, sizes, max_tiles=2048)
        for n in tiles:
            got = cache(packs[n][0][0]).clone()
            assert torch.equal(got, eager(packs[n][0][0])), n
        for n in (1201, 700, 333, 700):
            got = cache(packs[n][1][0]).clone()
            assert torch.equal(got, eager(packs[n][1][0])), n
        assert (cache.hits, cache.misses) == (4, 3)
        before = cache(packs[333][1][0]).clone()
        state = m.state_dict()
        state["encoder.layers.4.ffn.fc1.weight"] = state["encoder.layers.4.ffn.fc1.weight"] * 1.05
        m.load_state_dict(state)
        after = cache(packs[333][1][0]).clone()
        assert not torch.equal(after, before)
        assert torch.equal(after, eager(packs[333][1][0]))
        assert all(p.grad is None for p in m.parameters())
