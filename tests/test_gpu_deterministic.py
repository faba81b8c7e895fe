"""Deterministic mode on the B200 (``config.deterministic()``): the kernels that reduce gradients in a fixed order, held to
float64 references and to bitwise repeatability, and whole training steps that must give the same bits in every run.

Kernels: the deterministic dilated-attention backward (impl 4) against a float64 reference built on the device from the
same bf16 q / k / v / dO and the same lse / delta; a structural check that its branch order is fixed (one-branch runs
summed in branch order equal the five-branch run bit for bit); cross-attention and the three column reductions.

Steps: every run is a fresh process (this file is its own driver: ``python tests/test_gpu_deterministic.py OUT.pt
MODEL``), so nothing a first run leaves behind (allocator state, cached plans) can make a second run agree by accident.
"""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from modaltune_b200 import config, ops  # noqa: E402
from modaltune_b200.slide_encoder import DILATED_RATIO, optimal_segment_lengths  # noqa: E402
from tests.dilated_ref64 import bwd_ref64  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda"


def assert_bitwise_equal(a, b, what=""):
    """Same shape and the same bits in every element (NaN payloads and signed zeros included)."""
    assert a.shape == b.shape, (what, a.shape, b.shape)
    ai = a.detach().contiguous().view(torch.int32 if a.element_size() == 4 else torch.int16)
    bi = b.detach().contiguous().view(torch.int32 if b.element_size() == 4 else torch.int16)
    n = int((ai != bi).sum())
    assert n == 0, f"{what}: {n} elements differ"


def _one_ulp(t):
    """t with one element moved by one ulp."""
    t = t.detach().clone()
    flat = t.view(-1)
    i = flat.numel() // 2
    flat[i] = torch.nextafter(flat[i:i + 1], torch.full_like(flat[i:i + 1], float("inf")))[0]
    return t


def test_bitwise_helper_negative_control():
    x = torch.randn(1000, device=DEV)
    assert_bitwise_equal(x, x.clone())
    with pytest.raises(AssertionError):
        assert_bitwise_equal(x, _one_ulp(x))
    y = torch.randn(64, device=DEV).to(torch.bfloat16)
    with pytest.raises(AssertionError):
        assert_bitwise_equal(y, _one_ulp(y))


def within_abs_terms(got, ref64, abs_terms, bound, what=""):
    """|got - ref| <= bound * (sum of absolute terms) per element."""
    err = float(((got.double() - ref64).abs() / (abs_terms + 1e-30)).max())
    assert err <= bound, (what, err, bound)
    return err


def test_within_abs_terms_negative_control():
    x = torch.randn(100, 50, device=DEV, dtype=torch.float64)
    ref, terms = x.sum(0), x.abs().sum(0)
    within_abs_terms(x.float().sum(0), ref, terms, 1e-5)
    with pytest.raises(AssertionError):
        within_abs_terms(x.float().sum(0) + 1e-3 * terms.float(), ref, terms, 1e-5)


# ---------------------------------------------------------------------------------------------------------------------
# dilated attention backward, impl 4
# ---------------------------------------------------------------------------------------------------------------------
SIZES = [130, 1200, 5793, 10001, 32769]


def _dilated_inputs(N, sl=None, ratios=None):
    sl = sl or optimal_segment_lengths()
    ratios = ratios or DILATED_RATIO
    geom = ops.Geometry.get(N, sl, ratios)
    g = torch.Generator().manual_seed(N + 2)
    qkv = torch.zeros(geom.n_alloc, 2304)
    qkv[:N] = torch.randn(N, 2304, generator=g) * 1.5
    qkv = qkv.to(torch.bfloat16).to(DEV)
    gamma = (1 + 0.1 * torch.randn(768, generator=g)).to(DEV)
    beta = (0.1 * torch.randn(768, generator=g)).to(DEV)
    dy = torch.randn(N, 768, generator=g).to(DEV)
    o, l = ops.dilated_attn_fwd(geom, qkv, 3)
    _, _, lse, m, r = ops.dilated_merge_ln_fwd(geom, o, l, gamma, beta)
    dattn, delta = ops.dilated_merge_ln_bwd(geom, dy, o, l, gamma, m, r)
    return geom, qkv, dattn, lse, delta


@pytest.mark.parametrize("N", SIZES)
def test_dilated_bwd_impl4_vs_float64_and_repeat(N):
    geom, qkv, dattn, lse, delta = _dilated_inputs(N)
    a = ops.dilated_attn_bwd(geom, qkv, dattn, lse, delta, 4)
    b = ops.dilated_attn_bwd(geom, qkv, dattn, lse, delta, 4)
    torch.cuda.synchronize()
    assert torch.isfinite(a).all()
    assert_bitwise_equal(a, b, f"impl 4 repeat N={N}")
    ref, tabs = bwd_ref64(geom, qkv, dattn, lse, delta)
    for name, cols in (("dq", slice(0, 768)), ("dk", slice(768, 1536)), ("dv", slice(1536, 2304))):
        got, want = a[:, cols].double(), ref[:, cols]
        # per element: the bound of the tcgen05 backward (tests/test_gpu_dilated_sm100_ref64.py)
        within_abs_terms(got, want, tabs[:, cols], 2.0 ** -7, name)
        # the bars of the tcgen05 backward tests of impls 1 / 2 (tests/test_gpu_kernels.py)
        e = float((got - want).abs().max() / want.abs().max())
        assert e < 3e-2, (name, e)
        cos = torch.nn.functional.cosine_similarity(got.flatten(), want.flatten(), dim=0)
        assert float(cos) > 0.9995, (name, float(cos))


@pytest.mark.parametrize("N", SIZES)
def test_dilated_bwd_impl4_branch_order_is_fixed(N):
    """Each branch alone (a one-branch geometry, the full merged lse, that branch's delta) summed in branch order with
    fp32 adds equals the five-branch call bit for bit: every element gets one addition per branch, in branch order."""
    geom, qkv, dattn, lse, delta = _dilated_inputs(N)
    full = ops.dilated_attn_bwd(geom, qkv, dattn, lse, delta, 4)
    acc = torch.zeros_like(full)
    boff = 0
    for sl, r in zip(geom.segment_lengths, geom.ratios):
        g1 = ops.Geometry.get(N, [sl], [r])
        n = N * (16 // r)
        acc = acc + ops.dilated_attn_bwd(g1, qkv, dattn, lse, delta[boff: boff + n].contiguous(), 4)
        boff += n
    torch.cuda.synchronize()
    assert_bitwise_equal(acc, full, f"branch sum N={N}")


def test_dilated_bwd_impl4_rows_past_m_get_nothing():
    """N = 5793: branch 1 (segment 5792, dilation 2) has m = 2896 slots, so query tile 22 of segment 0 runs into the
    one-position segment 1.  With that position's key and value zero, its own tile adds exactly 0 to its dQ: any
    non-zero there would have come from the tile of segment 0 that does not own it."""
    N = 5793
    geom, qkv, dattn, lse, delta = _dilated_inputs(N, [5792], [2])
    qkv = qkv.clone()
    qkv[5792, 768:] = 0
    dq = ops.dilated_attn_bwd(geom, qkv, dattn, lse, delta, 4)
    torch.cuda.synchronize()
    assert float(dattn[5792].abs().sum()) > 0 and float(qkv[5792, :768].float().abs().sum()) > 0
    assert float(dq[5792, :768].abs().max()) == 0.0
    assert float(dq[5790, :384].abs().max()) > 0.0     # the last real query of segment 0 (residue 0) is written


# ---------------------------------------------------------------------------------------------------------------------
# cross-attention backward, deterministic
# ---------------------------------------------------------------------------------------------------------------------
def _cross_ref64(q, k, v, d_o, heads=12):
    q64, k64, v64 = (t.detach().double().requires_grad_(True) for t in (q, k, v))
    lq, lk = q.shape[0], k.shape[0]
    qh, kh, vh = q64.view(lq, heads, 16).transpose(0, 1), k64.view(lk, heads, 16).transpose(0, 1), v64.view(lk, heads, 16).transpose(0, 1)
    o = torch.softmax(qh @ kh.transpose(1, 2) / 4.0, -1) @ vh
    o.transpose(0, 1).reshape(lq, heads * 16).backward(d_o.double())
    return q64.grad, k64.grad, v64.grad


@pytest.mark.parametrize("lq,lk", [(10000, 66), (66, 10000)])
@pytest.mark.parametrize("layout", ["separate", "packed384", "packed1152"])
def test_cross_attn_bwd_deterministic(lq, lk, layout):
    g = torch.Generator().manual_seed(lq + 3 * lk)
    q, d_o = torch.randn(lq, 192, generator=g).to(DEV), torch.randn(lq, 192, generator=g).to(DEV)
    if layout == "separate":
        k, v = torch.randn(lk, 192, generator=g).to(DEV), torch.randn(lk, 192, generator=g).to(DEV)
    else:
        w = 384 if layout == "packed384" else 1152
        buf = torch.randn(lk, w, generator=g).to(DEV)
        k, v = buf[:, w - 384: w - 192], buf[:, w - 192:]
    o, lse = ops.cross_attn_fwd(q, k, v, 12, impl=1)
    with config.using(deterministic=True):
        r1 = ops.cross_attn_bwd(q, k, v, o, d_o, lse, 12, impl=1, packed_kv=layout != "separate")
        r2 = ops.cross_attn_bwd(q, k, v, o, d_o, lse, 12, impl=1, packed_kv=layout != "separate")
    torch.cuda.synchronize()
    refs = _cross_ref64(q, k, v, d_o)
    scale = lambda ref: max(float(ref.abs().max()), 0.1 * float(d_o.abs().max()))
    for name, a, b, ref in zip(("dq", "dk", "dv"), r1, r2, refs):
        assert_bitwise_equal(a, b, name)
        # the impl-1 bound of tests/test_gpu_kernels.py::test_cross_attention_tensor_core
        assert float((a.double() - ref).abs().max()) < 5e-3 * scale(ref), name


# ---------------------------------------------------------------------------------------------------------------------
# column reductions of the adapter's weight gradients
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows", [1, 1200, 10001])
def test_layernorm_bwd_weight_grads_deterministic(rows):
    g = torch.Generator().manual_seed(rows)
    dy, x = torch.randn(rows, 768, generator=g).to(DEV), torch.randn(rows, 768, generator=g).to(DEV)
    gamma = torch.randn(768, generator=g).to(DEV)
    mean, rstd = x.mean(1), (x.var(1, unbiased=False) + 1e-5).rsqrt()
    with config.using(deterministic=True):
        _, dg1, db1 = ops.layernorm_bwd(dy, x, gamma, mean, rstd, torch.float32, want_wgrad=True)
        _, dg2, db2 = ops.layernorm_bwd(dy, x, gamma, mean, rstd, torch.float32, want_wgrad=True)
    assert_bitwise_equal(dg1, dg2, "dgamma")
    assert_bitwise_equal(db1, db2, "dbeta")
    xh = (x.double() - mean.double()[:, None]) * rstd.double()[:, None]
    t = dy.double() * xh
    within_abs_terms(dg1, t.sum(0), t.abs().sum(0), 1e-5, "dgamma")
    within_abs_terms(db1, dy.double().sum(0), dy.double().abs().sum(0), 1e-5, "dbeta")


@pytest.mark.parametrize("rows", [1, 1200, 10000])
def test_gated_residual_bwd_deterministic(rows):
    g = torch.Generator().manual_seed(rows + 1)
    dy, a, b = (torch.randn(rows, 768, generator=g).to(DEV) for _ in range(3))
    gate = torch.randn(768, generator=g).to(DEV)
    with config.using(deterministic=True):
        r1 = ops.gated_residual_bwd(dy, a, b, gate, want_dysum=True)
        r2 = ops.gated_residual_bwd(dy, a, b, gate, want_dysum=True)
    for name, x1, x2 in zip(("da", "db", "dgate", "dysum"), r1, r2):
        assert_bitwise_equal(x1, x2, name)
    t = dy.double() * (a.double() + b.double())
    within_abs_terms(r1[2], t.sum(0), t.abs().sum(0), 1e-5, "dgate")
    within_abs_terms(r1[3], dy.double().sum(0), dy.double().abs().sum(0), 1e-5, "dysum")


@pytest.mark.parametrize("rows,cols", [(10000, 384), (10000, 192), (1024, 768), (40001, 768)])
def test_colsum_deterministic(rows, cols):
    g = torch.Generator().manual_seed(rows + cols)
    x = torch.randn(rows, cols + 8, generator=g).to(DEV)[:, :cols]
    with config.using(deterministic=True):
        s1, s2 = ops.colsum(x), ops.colsum(x)
    assert_bitwise_equal(s1, s2, "colsum")
    within_abs_terms(s1, x.double().sum(0), x.double().abs().sum(0), 1e-5, "colsum")


def test_deterministic_mode_selects_impl4_and_simt_raises():
    with config.using(deterministic=True):
        assert ops.dilated_bwd_impl(config.attn_impl("bwd")) == 4 and config.attn_impl("fwd") == config.AUTO_IMPL["fwd"]
        geom, qkv, dattn, lse, delta = _dilated_inputs(130)
        with pytest.raises(RuntimeError, match="deterministic"):
            ops.dilated_attn_bwd(geom, qkv, dattn, lse, delta, 0)


# ---------------------------------------------------------------------------------------------------------------------
# whole steps, each run in a fresh process
# ---------------------------------------------------------------------------------------------------------------------
def _run_driver(tmp_path, name, model, env_extra, torch_flag=False):
    out = str(tmp_path / f"{name}.pt")
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8", **env_extra)
    cmd = [sys.executable, os.path.abspath(__file__), out, model] + (["torch_flag"] if torch_flag else [])
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-6000:]
    return torch.load(out)


def _compare_runs(a, b, what):
    keys = [k for k in a if not k.startswith("meta")]
    assert keys == [k for k in b if not k.startswith("meta")]
    for k in keys:
        assert_bitwise_equal(a[k], b[k], f"{what}: {k}")


@pytest.mark.parametrize("model", ["toy", "full"])
def test_steps_are_bitwise_reproducible(tmp_path, model):
    r1 = _run_driver(tmp_path, "a", model, {"MODALTUNE_B200_DETERMINISTIC": "1"})
    r2 = _run_driver(tmp_path, "b", model, {"MODALTUNE_B200_DETERMINISTIC": "1"})
    _compare_runs(r1, r2, f"{model}: two runs")
    r3 = _run_driver(tmp_path, "c", model, {"MODALTUNE_B200_DETERMINISTIC": "0"}, torch_flag=True)
    _compare_runs(r1, r3, f"{model}: env switch vs torch.use_deterministic_algorithms")
    # within one process: eager and graph replay give the same bits (eval: train mode draws its dropout masks from
    # a different generator offset inside the graph, so there only run-to-run equality is asked for)
    for k in ("loss", "logits", "grads"):
        for i in (0, 1):
            assert_bitwise_equal(r1[f"eval/eager/{i}/{k}"], r1[f"eval/graph/{i}/{k}"], f"{model} eager vs graph: {k}")
        assert_bitwise_equal(r1[f"eval/eager/0/{k}"], r1[f"eval/cache/0/{k}"], f"{model} eager vs graph cache: {k}")
    assert r1["meta/recaptured"].item() == 1
    # accuracy: the deterministic step against the default step (the bar of the DESIGN.md A / B switches)
    lg, lg0 = r1["eval/eager/0/logits"].double(), r1["meta/default/logits"].double()
    assert float((lg - lg0).abs().max() / lg0.abs().max()) < 5e-3
    g, g0 = r1["eval/eager/0/grads"].double(), r1["meta/default/grads"].double()
    assert float(g @ g0 / (g.norm() * g0.norm())) > 0.9999


def _driver(out, model_kind, torch_flag):
    """One process: eager / GraphedStep / GraphCache steps in eval() and train() (two AdamW steps) with the same seeds."""
    from modaltune_b200 import synthetic, train_step
    from tests import helpers

    if torch_flag:
        torch.use_deterministic_algorithms(True)
    assert config.deterministic()
    dev = torch.device("cuda")
    torch.manual_seed(0)
    groups = helpers.SMALL_GROUPS if model_kind == "toy" else None
    tiles = (1300, 900) if model_kind == "toy" else (10000, 6000)
    model = helpers.build_model(groups, device=dev)
    proj = helpers.build_projector(0, dev)
    params = [p for p in model.parameters() if p.requires_grad]
    res = {}

    def record(tag, loss, logits):
        res[f"{tag}/loss"] = loss.detach().float().reshape(1).cpu()
        res[f"{tag}/logits"] = logits.detach().float().cpu()
        res[f"{tag}/grads"] = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).detach().reshape(-1)
                                         for p in params]).cpu()

    slides = [synthetic.synthetic_slide(t, seed=11 + i, group_sizes=groups) for i, t in enumerate(tiles)]
    dslide = train_step.slide_to_device(slides[0], dev)
    host = [train_step.pack_host_slide(s) for s in slides]
    flat = train_step.FlatGradAllReduce(params)
    init = [p.detach().clone() for p in params]

    def reset():
        with torch.no_grad():
            for p, p0 in zip(params, init):
                p.copy_(p0)

    for mode in ("eval", "train"):
        model.train(mode == "train")
        # eager: two steps (train: AdamW on the gradients)
        reset()
        opt = torch.optim.AdamW(params, lr=1e-4)
        torch.manual_seed(1)
        for i in range(2):
            flat.zero()
            model.zero_grad()
            loss, logits = train_step.forward_backward(model, proj, dslide)
            torch.cuda.synchronize()
            record(f"{mode}/eager/{i}", loss, logits)
            if mode == "train":
                opt.step()
                res[f"{mode}/eager/{i}/params"] = torch.cat([p.detach().reshape(-1) for p in params]).cpu()
        # the same two steps as graph replays
        reset()
        opt = torch.optim.AdamW(params, lr=1e-4)
        torch.manual_seed(1)
        step = train_step.GraphedStep(model, proj, {k: v.to(dev) for k, v in host[0][0].items()}, host[0][1], flat,
                                      warmup=1)
        torch.manual_seed(1)
        for i in range(2):
            loss, logits = step(host[0][0])
            torch.cuda.synchronize()
            record(f"{mode}/graph/{i}", loss, logits)
            if mode == "train":
                opt.step()
                res[f"{mode}/graph/{i}/params"] = torch.cat([p.detach().reshape(-1) for p in params]).cpu()
        if mode == "eval":
            # flipping the switch makes the step capture again
            g0 = step.graph
            with config.using(deterministic=False):
                if not torch.are_deterministic_algorithms_enabled():
                    step(host[0][0])
            res["meta/recaptured"] = torch.tensor(int(step.graph is not g0 or torch.are_deterministic_algorithms_enabled()))
            del step
            # a graph cache over two shapes: the first shape again, then the second
            reset()
            cache = train_step.GraphCache(model, proj, flat, host[0][1], max_tiles=max(tiles))
            for i, (hp, _, _) in enumerate(host):
                loss, logits = cache(hp)
                torch.cuda.synchronize()
                record(f"{mode}/cache/{i}", loss, logits)
            del cache
    # the default (non-deterministic) step on the same inputs, for the accuracy comparison
    if not torch_flag:
        reset()
        model.eval()
        with config.using(deterministic=False):
            model.zero_grad()
            loss, logits = train_step.forward_backward(model, proj, dslide)
            torch.cuda.synchronize()
        res["meta/default/logits"] = logits.detach().float().cpu()
        res["meta/default/grads"] = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1)
                                               for p in params]).cpu()
    else:
        res["meta/recaptured"] = torch.tensor(1)
    torch.save(res, out)


if __name__ == "__main__":
    _driver(sys.argv[1], sys.argv[2], len(sys.argv) > 3 and sys.argv[3] == "torch_flag")
