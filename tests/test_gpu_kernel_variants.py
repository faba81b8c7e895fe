"""The kernel variants the default bf16 eval step runs (``mt_linear_sm100`` FFN epilogues, ``mt_ffn_bwd_prep``, branch
merge + LayerNorm at bench sizes, cross-attention on a column slice of the shared k | v projection, the gated-residual
and in-place LayerNorm backward of the Injector), each held to a plain float64 reference of the same operation.

Every reference is computed on the device in float64 from the exact operands the kernel saw (the bf16-rounded A and W,
the rounded gelu / gelu', the fp32 statistics handed in), so the tolerances only have to cover fp32 accumulation and one
rounding of the output: bf16 outputs are checked in units of one bf16 ulp of the float64 value, with an absolute floor
where that value is ~0 and the fp32 error of what feeds it is larger than its ulp.  TF32 never enters a reference:
nothing below multiplies fp32 matrices with torch.  Every position of every output is checked, not a sample of rows.
Each group ends with a negative control: the same assertion helper run against a deliberately wrong reference must fail.

``pytest -s`` prints the largest error each check measured next to its bound.
"""
import types

import pytest
import torch
import torch.nn.functional as F

from modaltune_b200 import _lib, ops
from modaltune_b200.slide_encoder import DILATED_RATIO, LongNetEncoderLayer, optimal_segment_lengths

pytestmark = pytest.mark.gpu
DEV = "cuda"
F64 = torch.float64
BF16 = torch.bfloat16
EPS = 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# assertion helpers
# ---------------------------------------------------------------------------------------------------------------------
def _report(name, value, bound):
    print(f"[measured] {name}: {value:.3g} (bound {bound:.3g})")


def bf16_ulp(ref):
    """Spacing of bf16 numbers (8 significant bits) at |ref|; 0 where ref is 0."""
    a = ref.abs()
    return torch.where(a > 0, torch.exp2(torch.floor(torch.log2(a)) - 7), torch.zeros_like(a))


def assert_ulps(name, got, ref, n, floor):
    """max |got - ref| / (ulp_bf16(ref) + floor) <= n.  ``floor`` (scalar or elementwise, > 0) is the absolute error of
    what feeds the value, which dominates only where the float64 value is ~0."""
    e = float(((got.double() - ref).abs() / (bf16_ulp(ref) + floor)).max())
    _report(name, e, n)
    assert e <= n, f"{name}: {e:.3g} bf16 ulp (+ floor) > {n}"


def assert_within(name, got, ref, bound, scale):
    """max |got - ref| / scale <= bound; ``scale`` (scalar or elementwise) is the size of what the value is formed from,
    e.g. the sum of |terms| of a reduction, so that a sum that cancels to ~0 is not held to a relative tolerance."""
    e = float(((got.double() - ref).abs() / scale).max())
    _report(name, e, bound)
    assert e <= bound, f"{name}: {e:.3g} > {bound:.3g}"


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


# ---------------------------------------------------------------------------------------------------------------------
# A. the FFN chain on mt_linear_sm100: fc1 + GELU + slab statistics, fc2 with the LayerNorm folded in, the fused
#    GELU' . LayerNorm' backward epilogue, mt_ffn_bwd_prep, and the whole FFN half-layer
# ---------------------------------------------------------------------------------------------------------------------
# row-tile (128) and CTA-pair (256) tails, and the 10k / 40k-token sizes of the benchmark configurations
FFN_ROWS = [1, 127, 128, 129, 255, 256, 257, 513, 10001, 40001]
FFN = 3072


def _ffn_operands(M, seed, x1_scale=1.0):
    g = _gen(seed)
    r = lambda *s: torch.randn(*s, generator=g, device=DEV)
    op = types.SimpleNamespace()
    op.a = r(M, 768).to(BF16)                                    # fc1's A operand (bf16 output of final_layer_norm)
    op.w1 = (r(FFN, 768) * 0.04).to(BF16)
    # column offsets from -7.5 to 7.5 on top of a unit-size product: every row meets gelu's minimum (h = -0.75, where
    # gelu' changes sign), its most negative slope (h = -1.5) and both saturated tails (|h| > 6)
    op.b1 = torch.linspace(-7.5, 7.5, FFN, device=DEV)[torch.randperm(FFN, generator=g, device=DEV)]
    w2 = r(768, FFN) * 0.02
    gam, bet, b2 = 1 + 0.1 * r(FFN), 0.1 * r(FFN), 0.1 * r(768)
    # the fold of ops.FrozenLayerWeights: W2' = W2 diag(gamma) in bf16, c1 = W2' 1 over the rounded W2', c2 = W2 beta + b2
    op.w2g = (w2 * gam).to(BF16)
    op.c1 = op.w2g.float().sum(1)
    op.c2 = (w2.double() @ bet.double() + b2.double()).float()
    op.x1 = r(M, 768) * x1_scale                                 # the FFN's residual input
    op.dy = r(M, 768)                                            # gradient of the layer output
    return op


def _fc1(op, impl, aux=True):
    """MT_EPI_GELU_STATS as the layer forward calls it (out_aux = gelu'(h), no fp32 h) or with the fp32 h instead."""
    M = op.a.shape[0]
    stats = torch.full((M, FFN // 128, 2), float("nan"), device=DEV)   # every slab partial must be written
    u = torch.empty((M, FFN), device=DEV, dtype=BF16)
    if aux:
        gd = torch.empty((M, FFN), device=DEV, dtype=BF16)
        ops.linear_sm100(op.a, op.w1, mode=_lib.MT_EPI_GELU_STATS, bias=op.b1, want_f32=False, out_bf16=u, out_aux=gd,
                         stats=stats, impl=impl)
        return u, gd, stats
    h, _ = ops.linear_sm100(op.a, op.w1, mode=_lib.MT_EPI_GELU_STATS, bias=op.b1, want_f32=True, out_bf16=u,
                            stats=stats, impl=impl)
    return u, h, stats


def _fc2(op, u, stats, impl):
    """MT_EPI_LN_RESIDUAL with the row statistics published, as the layer forward calls it."""
    M = u.shape[0]
    mean_f = torch.empty(M, device=DEV)
    rstd_f = torch.empty(M, device=DEV)
    y, _ = ops.linear_sm100(u, op.w2g, mode=_lib.MT_EPI_LN_RESIDUAL, residual=op.x1, stats=stats, col_c1=op.c1,
                            col_c2=op.c2, ln_cols=FFN, ln_mean_out=mean_f, ln_rstd_out=rstd_f, impl=impl)
    return y, mean_f, rstd_f


def _gelu_grad64(h):
    return 0.5 * (1 + torch.erf(h * 0.5 ** 0.5)) + h * torch.exp(-0.5 * h * h) * (2 * torch.pi) ** -0.5


def _ln_stats64(u):
    mean = u.mean(1)
    return mean, (u.var(1, unbiased=False) + EPS).rsqrt()


# The epilogue's erf is Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7) and cdf = (1 + erf) / 2 is formed in fp32, so far in
# the negative tail (h < -4, gelu(h) ~ 1e-5 and smaller) gelu and gelu' carry an ABSOLUTE error of ~|h| 1e-7 that is
# many ulps of their tiny values: that, not bf16 rounding, sets the floor there.
def _check_gelu_outputs(tag, u, gd, h):
    h64 = h.double()
    assert_ulps(f"{tag} u vs gelu(h)", u, F.gelu(h64), 1, floor=2.0 ** -21 * (1 + h64.abs()))
    assert_ulps(f"{tag} gelu' vs d gelu(h)/dh", gd, _gelu_grad64(h64), 1, floor=2.0 ** -21)


def _check_slab_stats(tag, stats, u):
    s = u.double().view(u.shape[0], FFN // 128, 128)
    assert_within(f"{tag} slab sum u", stats[..., 0], s.sum(2), 1e-5, s.abs().sum(2) + 1e-30)
    assert_within(f"{tag} slab sum u^2", stats[..., 1], s.square().sum(2), 1e-5, s.square().sum(2) + 1e-30)


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("M", FFN_ROWS)
def test_fc1_gelu_stats_epilogue(M, impl):
    op = _ffn_operands(M, seed=M)
    u, gd, stats = _fc1(op, impl)
    u2, h, stats2 = _fc1(op, impl, aux=False)
    # the auxiliary output changes nothing else the epilogue writes
    assert torch.equal(u, u2) and torch.equal(stats, stats2)
    # h against the float64 product of the same bf16 operands (fp32 accumulation over K = 768)
    h64 = op.a.double() @ op.w1.double().t() + op.b1.double()
    assert_within("fc1 h", h, h64, 1e-5, op.a.double().abs() @ op.w1.double().abs().t() + op.b1.double().abs())
    # gelu / gelu' against float64 at the fp32 h the epilogue computed (the same accumulator: bit-identical u above)
    _check_gelu_outputs("fc1", u, gd, h)
    # the slab partials are sums of the ROUNDED u
    _check_slab_stats("fc1", stats, u)


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("M", FFN_ROWS)
def test_fc2_layernorm_fold_epilogue(M, impl):
    op = _ffn_operands(M, seed=M + 1)
    u, _, stats = _fc1(op, impl)
    y, mean_f, rstd_f = _fc2(op, u, stats, impl)
    u64 = u.double()
    mean64, rstd64 = _ln_stats64(u64)
    assert_within("fc2 ln mean", mean_f, mean64, 1e-5, u64.abs().mean(1))
    assert_within("fc2 ln rstd", rstd_f, rstd64, 1e-5, rstd64)
    y64 = rstd64[:, None] * (u64 @ op.w2g.double().t() - mean64[:, None] * op.c1.double()) + op.c2.double() + op.x1.double()
    # relative to the size of the FFN branch of each row (the residual is added exactly, up to fp32 rounding)
    branch = (y64 - op.x1.double()).abs().amax(1, keepdim=True)
    assert_within("fc2 y", y, y64, 2e-4, branch)


def _fc2_dx_references(op, h, u, gd):
    """float64 references of MT_EPI_GELU_LN_BWD (the dX GEMM of fc2, W = (W2 diag gamma)^T) for dy rounded to bf16:
    the autograd of LN(gelu(h)) -> fc2 at the fp32 h, and the row vectors (mean, rstd, m1, m2) of both input forms."""
    dy16 = op.dy.to(BF16)
    w2g = op.w2g.double()
    gdn = dy16.double() @ w2g                                     # gamma_j dn_j
    h64 = h.double().requires_grad_(True)
    with torch.enable_grad():
        out = F.layer_norm(F.gelu(h64), (FFN,), eps=EPS) @ w2g.t()
        (dh64,) = torch.autograd.grad(out, h64, dy16.double())
    rowv = {}
    for form, u64 in (("h", F.gelu(h.double())), ("u", u.double())):
        mean, rstd = _ln_stats64(u64)
        uhat = (u64 - mean[:, None]) * rstd[:, None]
        rowv[form] = torch.stack([mean, rstd, gdn.mean(1), (gdn * uhat).mean(1)], 1).float().contiguous()
    # the written semantics of the in_u / in_g form (tests/cpu_kernels.linear_sm100, mode 5) on its exact operands
    mean, rstd, m1, m2 = (c[:, None] for c in rowv["u"].double().unbind(1))
    spec_u = gd.double() * rstd * (gdn - m1 - (u.double() - mean) * rstd * m2)
    return dy16, dh64, rowv, spec_u


def _fc2_dx(op, dy16, rowv, impl, h=None, u=None, gd=None):
    _, d = ops.linear_sm100(dy16, op.w2g.t().contiguous(), mode=_lib.MT_EPI_GELU_LN_BWD, residual=h, in_u=u, in_g=gd,
                            stats=rowv, want_f32=False, want_bf16=True, impl=impl)
    return d


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("M", FFN_ROWS)
def test_fc2_dx_gelu_layernorm_backward_epilogue(M, impl):
    op = _ffn_operands(M, seed=M + 2)
    u, gd, _ = _fc1(op, impl)
    _, h, _ = _fc1(op, impl, aux=False)
    dy16, dh64, rowv, spec_u = _fc2_dx_references(op, h, u, gd)
    d_h = _fc2_dx(op, dy16, rowv["h"], impl, h=h)                 # h through `residual`
    d_u = _fc2_dx(op, dy16, rowv["u"], impl, u=u, gd=gd)          # gelu / gelu' in bf16 from the forward epilogue
    # the error scale where the float64 value is ~0: fp32 accumulation of the dX GEMM and the cancellation inside
    # (acc - m1 - uhat m2), both proportional to the largest gradient (the scale() idiom of the cross-attention tests)
    top = float(dh64.abs().max())
    assert_ulps("fc2 dX (h form) vs float64 autograd", d_h, dh64, 1, floor=2.0 ** -16 * top)
    assert_ulps("fc2 dX (u, gelu' form) vs its spec", d_u, spec_u, 1, floor=2.0 ** -16 * top)
    # the u form rounds gelu and gelu' to bf16 before the epilogue reads them: one more ulp, and a wider floor
    assert_ulps("fc2 dX (u, gelu' form) vs float64 autograd", d_u, dh64, 2, floor=2.0 ** -12 * top)
    assert_ulps("fc2 dX u form vs h form", d_u, d_h.double(), 2, floor=2.0 ** -12 * top)


@pytest.mark.parametrize("x1_scale", [1.0, 100.0])
@pytest.mark.parametrize("M", FFN_ROWS)
def test_ffn_bwd_prep_on_forward_outputs(M, x1_scale):
    """m2 = dy . (y - x1 - c2) / C holds only because y IS the folded fc2 forward: hold it to the definition
    m2 = mean_j(gamma_j dn_j uhat_j) on real forward outputs, also with a residual stream 100x the FFN branch, where
    y - x1 - c2 cancels ~7 bits of y's fp32 mantissa: the same bound holds, because the rounding errors of y enter m2
    through a 768-term dot product with dy and average out."""
    op = _ffn_operands(M, seed=M + 3, x1_scale=x1_scale)
    u, _, stats = _fc1(op, 0)
    y, mean_f, rstd_f = _fc2(op, u, stats, 0)
    rowv, d16 = ops.ffn_bwd_prep(op.dy, y, op.x1, op.c1, op.c2, mean_f, rstd_f, FFN)
    assert torch.equal(d16, op.dy.to(BF16))
    assert torch.equal(rowv[:, 0], mean_f) and torch.equal(rowv[:, 1], rstd_f)
    gdn = d16.double() @ op.w2g.double()                          # gamma_j dn_j with dn = dy W2
    mean, rstd = _ln_stats64(u.double())
    t2 = gdn * (u.double() - mean[:, None]) * rstd[:, None]
    assert_within("ffn_bwd_prep m1", rowv[:, 2], gdn.mean(1), 1e-5, gdn.abs().mean(1))
    assert_within(f"ffn_bwd_prep m2 (x1 = {x1_scale:g} x branch)", rowv[:, 3], t2.mean(1), 1e-5, t2.abs().mean(1))


def _frozen_layer_weights(seed):
    """ops.FrozenLayerWeights of an encoder layer with seeded parameters (weights on the bf16 grid, as a checkpoint
    stored in bf16 would be) and the float64 copies the reference uses."""
    g = _gen(seed)
    layer = LongNetEncoderLayer(768, 16, FFN, optimal_segment_lengths(), DILATED_RATIO).to(DEV)
    with torch.no_grad():
        for name, p in layer.named_parameters():
            if name.endswith("weight") and p.dim() == 2:
                p.copy_((torch.randn(p.shape, generator=g, device=DEV) * p.shape[1] ** -0.5).to(BF16))
            elif "norm" in name or "ln" in name:
                p.copy_((1.0 if name.endswith("weight") else 0.0) + 0.1 * torch.randn(p.shape, generator=g, device=DEV))
            else:
                p.copy_(0.1 * torch.randn(p.shape, generator=g, device=DEV))
        layer.requires_grad_(False)
    return layer, ops.FrozenLayerWeights().refresh(layer, BF16)


def _ffn_half_layer(x1, W, dy):
    """The FFN half of _encoder_layer_forward_sm100 / _encoder_layer_backward_sm100, call for call (fused backward)."""
    N = x1.shape[0]
    h2, mean2, rstd2 = ops.layernorm_fwd(x1, W.ln2[0], W.ln2[1], BF16)
    stats = torch.empty((N, W.w_1.shape[0] // 128, 2), device=DEV)
    f1 = torch.empty((N, W.w_1.shape[0]), device=DEV, dtype=BF16)
    u = torch.empty((N, W.w_1.shape[0]), device=DEV, dtype=BF16)
    ops.linear_sm100(h2, W.w_1, mode=_lib.MT_EPI_GELU_STATS, bias=W.b_1, want_f32=False, out_bf16=u, out_aux=f1, stats=stats)
    mean_f = torch.empty(N, device=DEV)
    rstd_f = torch.empty(N, device=DEV)
    y, _ = ops.linear_sm100(u, W.w_2g, mode=_lib.MT_EPI_LN_RESIDUAL, residual=x1, stats=stats, col_c1=W.c1_2, col_c2=W.c2_2,
                            ln_cols=W.w_2g.shape[1], ln_mean_out=mean_f, ln_rstd_out=rstd_f)
    rowv, d_f2 = ops.ffn_bwd_prep(dy, y, x1, W.c1_2, W.c2_2, mean_f, rstd_f, W.w_2g.shape[1])
    _, d_f1 = ops.linear_sm100(d_f2, W.w_2g_t, mode=_lib.MT_EPI_GELU_LN_BWD, in_u=u, in_g=f1, stats=rowv, want_f32=False,
                               want_bf16=True)
    dh2, _ = ops.linear_sm100(d_f1, W.w_1_t)
    dx1, _, _ = ops.layernorm_bwd(dh2, x1, W.ln2[0], mean2, rstd2, torch.float32, residual=dy, bf16_twin=True)
    return y, dx1


@pytest.mark.parametrize("M", [1, 127, 257, 10001, 40001])
def test_ffn_half_layer_end_to_end(M):
    """y = x1 + fc2(LN(gelu(fc1(LN(x1))))) and its dX through the product's calls, against float64 with the model's
    parameters, row by row.  The bounds are the bf16 chain's (LN output, u, W2 diag(gamma), dy and d_f1 are rounded)."""
    layer, W = _frozen_layer_weights(M + 4)
    g = _gen(M + 5)
    x1 = torch.randn(M, 768, generator=g, device=DEV)
    dy = torch.randn(M, 768, generator=g, device=DEV)
    y, dx1 = _ffn_half_layer(x1, W, dy)
    d = lambda p: p.detach().double()
    ffn, ln2 = layer.ffn, layer.final_layer_norm
    x64 = x1.double().requires_grad_(True)
    with torch.enable_grad():
        h = F.layer_norm(x64, (768,), d(ln2.weight), d(ln2.bias), EPS) @ d(ffn.fc1.weight).t() + d(ffn.fc1.bias)
        n = F.layer_norm(F.gelu(h), (FFN,), d(ffn.ffn_layernorm.weight), d(ffn.ffn_layernorm.bias), EPS)
        branch = n @ d(ffn.fc2.weight).t() + d(ffn.fc2.bias)
        (dx64,) = torch.autograd.grad(x64 + branch, x64, dy.double())
    assert_within("FFN half-layer y, per row", y, x64.detach() + branch.detach(), 2e-2,
                  branch.detach().abs().amax(1, keepdim=True))
    dbranch = dx64 - dy.double()
    assert_within("FFN half-layer dX, per row", dx1, dx64, 3e-2, dbranch.abs().amax(1, keepdim=True))


def test_ffn_negative_controls():
    """The helpers and bounds above fail on a kernel that is subtly wrong: gelu' replaced by h, slab statistics one slab
    off, m2 = 0 in the prep row vector and in the backward epilogue's reference."""
    M = 513
    op = _ffn_operands(M, seed=M)
    u, gd, stats = _fc1(op, 2)
    _, h, _ = _fc1(op, 2, aux=False)
    h64 = h.double()
    with pytest.raises(AssertionError):
        assert_ulps("control: h as gelu'", gd, h64, 1, floor=2.0 ** -21)
    with pytest.raises(AssertionError):
        _check_slab_stats("control: slabs shifted", stats.roll(1, dims=1), u)
    y, mean_f, rstd_f = _fc2(op, u, stats, 2)
    rowv, d16 = ops.ffn_bwd_prep(op.dy, y, op.x1, op.c1, op.c2, mean_f, rstd_f, FFN)
    t2 = (d16.double() @ op.w2g.double()) * (u.double() - mean_f.double()[:, None]) * rstd_f.double()[:, None]
    with pytest.raises(AssertionError):
        assert_within("control: m2 = 0", rowv[:, 3], torch.zeros_like(t2[:, 0]), 1e-5, t2.abs().mean(1))
    dy16, dh64, rowv64, _ = _fc2_dx_references(op, h, u, gd)
    d_h = _fc2_dx(op, dy16, rowv64["h"], 2, h=h)
    no_m2 = rowv64["h"].clone()
    no_m2[:, 3] = 0
    d_wrong = _fc2_dx(op, dy16, no_m2, 2, h=h)
    top = float(dh64.abs().max())
    with pytest.raises(AssertionError):   # the epilogue run without m2 against the true gradient
        assert_ulps("control: dX with m2 = 0", d_wrong, dh64, 1, floor=2.0 ** -16 * top)
    assert_ulps("control baseline: dX", d_h, dh64, 1, floor=2.0 ** -16 * top)


# ---------------------------------------------------------------------------------------------------------------------
# B. branch merge + inner_attn_ln (mt_dilated_merge_ln_fwd / _bwd) at bench geometries
# ---------------------------------------------------------------------------------------------------------------------
MERGE_GEOMS = [(10001, None), (32769, None), (40001, None),
               # whole-tile edge cases of the tcgen05 tests (last segments with 1 / 128 / 129 real slots, all-padding tails)
               (1153, None), (2177, [1024, 2048, 4096, 8192, 16384]), (8193, None), (16385, None),
               (4224, [512, 1024, 2048, 4096, 8192]), (12289, [4096, 4096, 8192, 8192, 16384]),
               # no segment length a power of two: p % g through the float reciprocal of g at every branch
               (40001, [24, 96, 1448, 5792, 23168])]


def _merge_inputs(geom, seed):
    g = _gen(seed)
    o_br = torch.randn(geom.o_elems, generator=g, device=DEV).to(BF16)
    # most branch LSEs within a few nats of each other; one entry in ten lifted by 35 nats, so that it dominates the
    # others by more than 30 (weights of e^-30 and below next to it)
    lse_br = (6 + 2 * torch.randn(geom.lse_elems, generator=g, device=DEV)
              + 35 * (torch.rand(geom.lse_elems, generator=g, device=DEV) < 0.1).float())
    gamma = 1 + 0.1 * torch.randn(768, generator=g, device=DEV)
    beta = 0.1 * torch.randn(768, generator=g, device=DEV)
    dy = torch.randn(geom.n_tokens, 768, generator=g, device=DEV)
    return o_br, lse_br, gamma, beta, dy


def _merge_ref(geom, o_br, lse_br, owner_shift=0, chunk=8192):
    """float64 merge from the layout of include/modaltune_b200.h: branch b (segment g = min(sl, N), dilation r) owns
    (p, h) iff (p % g) % r == h r / H, and keeps it in slot h % (H / r) of row p of its compact [N][H/r] block.
    -> attn [N, 768], lse [N, 16]; built chunk by chunk over positions."""
    N, H, D = geom.n_tokens, geom.heads, geom.head_dim
    attn = torch.empty((N, H * D), device=DEV, dtype=F64)
    lse = torch.empty((N, H), device=DEV, dtype=F64)
    hs = torch.arange(H, device=DEV)
    for p0 in range(0, N, chunk):
        rows = slice(p0, min(N, p0 + chunk))
        p = torch.arange(rows.start, rows.stop, device=DEV)
        Ls, Os, o_off, l_off = [], [], 0, 0
        for sl, r in zip(geom.segment_lengths, geom.ratios):
            g, hpb = min(sl, N), H // r
            ob = o_br[o_off:o_off + N * hpb * D].view(N, hpb, D)[rows].double()
            lb = lse_br[l_off:l_off + N * hpb].view(N, hpb)[rows].double()
            own = (((p + owner_shift) % g) % r)[:, None] == (hs * r // H)[None, :]
            Ls.append(torch.where(own, lb[:, hs % hpb], float("-inf")))
            Os.append(ob[:, hs % hpb])
            o_off += N * hpb * D
            l_off += N * hpb
        L = torch.stack(Ls)
        w = torch.softmax(L, 0)
        attn[rows] = (w[..., None] * torch.stack(Os)).sum(0).reshape(-1, H * D)
        lse[rows] = torch.logsumexp(L, 0)
    return attn, lse


def _delta_ref(geom, dattn, o_br):
    """delta_b[p, slot] = dattn[p, head, :] . o_b[p, slot, :] over the heads branch b's slots hold, in the compact layout,
    and the sum of |terms| of each dot product."""
    N, H, D = geom.n_tokens, geom.heads, geom.head_dim
    d3 = dattn[:N].double().view(N, H, D)
    p = torch.arange(N, device=DEV)
    outs, scales, o_off = [], [], 0
    for sl, r in zip(geom.segment_lengths, geom.ratios):
        g, hpb = min(sl, N), H // r
        ob = o_br[o_off:o_off + N * hpb * D].view(N, hpb, D).double()
        heads = ((p % g) % r)[:, None] * hpb + torch.arange(hpb, device=DEV)[None, :]
        t = d3[p[:, None], heads] * ob
        outs.append(t.sum(-1).reshape(-1))
        scales.append(t.abs().sum(-1).reshape(-1))
        o_off += N * hpb * D
    return torch.cat(outs), torch.cat(scales)


def _check_merge_attn(tag, attn, attn64, o_br):
    # fp32 merge of <= 5 branch rows: a few fp32 roundings of max |o| where attn cancels to ~0
    assert_ulps(f"{tag} attn", attn, attn64, 1, floor=2.0 ** -18 * float(o_br.float().abs().max()))


@pytest.mark.parametrize("N,sl", MERGE_GEOMS)
def test_merge_layernorm_at_bench_geometries(N, sl):
    geom = ops.Geometry.get(N, sl or optimal_segment_lengths(), DILATED_RATIO)
    o_br, lse_br, gamma, beta, dy = _merge_inputs(geom, N + len(sl or []))
    y, attn, lse, mean, rstd = ops.dilated_merge_ln_fwd(geom, o_br, lse_br, gamma, beta, want_attn=True)
    # as the layer backward calls it: fp32 dy (the out_proj dX GEMM's output), bf16 branch outputs
    dattn, delta = ops.dilated_merge_ln_bwd(geom, dy, o_br, lse_br, gamma, mean, rstd)
    attn64, lse64 = _merge_ref(geom, o_br, lse_br)
    _check_merge_attn(f"merge N={N}", attn, attn64, o_br)
    assert_within(f"merge N={N} lse", lse, lse64, 1e-6, lse64.abs() + 1)
    mean64, rstd64 = _ln_stats64(attn64)
    assert_within(f"merge N={N} ln mean", mean, mean64, 1e-5, attn64.abs().mean(1))
    assert_within(f"merge N={N} ln rstd", rstd, rstd64, 1e-5, rstd64)
    xhat = (attn64 - mean64[:, None]) * rstd64[:, None]
    y64 = xhat * gamma.double() + beta.double()
    assert_ulps(f"merge N={N} y", y, y64, 1, floor=2.0 ** -16 * float(y64.abs().max()))
    gd = dy.double() * gamma.double()
    dattn64 = rstd64[:, None] * (gd - gd.mean(1, keepdim=True) - xhat * (gd * xhat).mean(1, keepdim=True))
    assert dattn.shape[0] == geom.n_alloc and not bool(dattn[N:].any())
    assert_ulps(f"merge N={N} dattn", dattn[:N], dattn64, 1, floor=2.0 ** -16 * float(dattn64.abs().max()))
    # delta is formed from the ROUNDED dattn the attention backward reads
    delta64, dscale = _delta_ref(geom, dattn, o_br)
    assert_within(f"merge N={N} delta_br", delta, delta64, 1e-5, dscale + 1e-30)


def test_merge_negative_control():
    """Ownership one position off moves every (position, head) of the dilated branches to a neighbour's owner."""
    geom = ops.Geometry.get(10001, optimal_segment_lengths(), DILATED_RATIO)
    o_br, lse_br, gamma, beta, _ = _merge_inputs(geom, 10001)
    _, attn, _, _, _ = ops.dilated_merge_ln_fwd(geom, o_br, lse_br, gamma, beta, want_attn=True)
    with pytest.raises(AssertionError):
        _check_merge_attn("control: owner off by one", attn, _merge_ref(geom, o_br, lse_br, owner_shift=1)[0], o_br)


# ---------------------------------------------------------------------------------------------------------------------
# C. cross-attention with k | v read as a column slice of the [Lk, 3 x 384] projection the last block's extractors share
# ---------------------------------------------------------------------------------------------------------------------
def _cross_ref(q, k, v, d_o, heads=12):
    qq, kk, vv = (t.double().requires_grad_(True) for t in (q, k, v))
    with torch.enable_grad():
        qh, kh, vh = (t.reshape(t.shape[0], heads, -1).transpose(0, 1) for t in (qq, kk, vv))
        s = qh @ kh.transpose(1, 2) / qh.shape[-1] ** 0.5
        lse = torch.logsumexp(s, -1)
        o = (torch.exp(s - lse[..., None]) @ vh).transpose(0, 1).reshape(q.shape)
        dq, dk, dv = torch.autograd.grad(o, [qq, kk, vv], d_o.double())
    return o.detach(), lse.t().detach(), dq, dk, dv


def _check_cross(tag, impl, got, ref, d_o):
    """The bounds of test_gpu_kernels: exact fp32 SIMT math (impl 0), TF32 operands (impl 1, gradients relative to the
    larger of the gradient and 0.1 |d_o|)."""
    o, lse, dq, dk, dv = got
    o64, lse64, dq64, dk64, dv64 = ref
    rel = lambda a, b: float((a.double() - b).abs().max() / b.abs().max())
    checks = [("o", rel(o, o64), 2e-5 if impl == 0 else 3e-3), ("lse", rel(lse, lse64), 1e-5 if impl == 0 else 1e-3)]
    for name, gr, r64 in (("dq", dq, dq64), ("dk", dk, dk64), ("dv", dv, dv64)):
        scale = max(float(r64.abs().max()), 0.1 * float(d_o.abs().max())) if impl == 1 else float(r64.abs().max())
        checks.append((name, float((gr.double() - r64).abs().max()) / scale, 5e-5 if impl == 0 else 5e-3))
    for name, e, bound in checks:
        _report(f"{tag} {name}", e, bound)
    bad = [(name, e, bound) for name, e, bound in checks if not e <= bound]
    assert not bad, f"{tag}: {bad}"


def _cross_run(q, k, v, d_o, impl):
    o, lse = ops.cross_attn_fwd(q, k, v, 12, impl=impl)
    dq, dk, dv = ops.cross_attn_bwd(q, k, v, o, d_o, lse, 12, impl=impl, packed_kv=True)
    return o, lse, dq, dk, dv


@pytest.mark.parametrize("lk", [10001, 40001])
@pytest.mark.parametrize("lq", [1, 66, 333])
def test_cross_attention_on_a_column_slice_of_the_shared_kv_projection(lq, lk):
    g = _gen(lq * 7 + lk)
    q = torch.randn(lq, 192, generator=g, device=DEV)
    d_o = torch.randn(lq, 192, generator=g, device=DEV)
    kv3 = torch.randn(lk, 3 * 384, generator=g, device=DEV)      # ldkv = 1152
    for off in (0, 384, 768):
        k, v = kv3[:, off:off + 192], kv3[:, off + 192:off + 384]
        kc, vc = k.contiguous(), v.contiguous()
        ref = _cross_ref(q, kc, vc, d_o)
        for impl in (0, 1):
            got = _cross_run(q, k, v, d_o, impl)
            flat = _cross_run(q, kc, vc, d_o, impl)
            # the split-K forward combines its partials in a fixed order, and dk / dv (one thread per key, loop over
            # the few queries) are plain stores: bit-identical.  dq of few queries over many keys is split over the keys
            # and reduced with fp32 atomics in arbitrary order, so only the rounding of those adds may differ.
            for name, a, b in zip(("o", "lse", "dk", "dv"), got[:2] + got[3:], flat[:2] + flat[3:]):
                assert torch.equal(a, b), (off, impl, name)
            assert float((got[2] - flat[2]).abs().max()) <= 1e-6 * float(flat[2].abs().max()), (off, impl)
            _check_cross(f"cross lq={lq} lk={lk} off={off} impl={impl}", impl, got, ref, d_o)


def test_cross_attention_negative_control():
    """k read from column offset 384 instead of 0 (the next extractor's k | v)."""
    g = _gen(5)
    lq, lk = 66, 10001
    q, d_o = torch.randn(lq, 192, generator=g, device=DEV), torch.randn(lq, 192, generator=g, device=DEV)
    kv3 = torch.randn(lk, 3 * 384, generator=g, device=DEV)
    got = _cross_run(q, kv3[:, :192], kv3[:, 192:384], d_o, 1)
    with pytest.raises(AssertionError):
        _check_cross("control: k at offset 384", 1, got, _cross_ref(q, kv3[:, 384:576], kv3[:, 192:384], d_o), d_o)


# ---------------------------------------------------------------------------------------------------------------------
# D. the Injector's small kernels: gated-residual backward column sums, LayerNorm backward with residual aliasing dx
# ---------------------------------------------------------------------------------------------------------------------
def _gated_operands(rows, bdt, seed):
    g = _gen(seed)
    a, b, dy = (torch.randn(rows, 768, generator=g, device=DEV) for _ in range(3))
    gate = 0.5 * torch.randn(768, generator=g, device=DEV)
    return a, b.to(bdt), gate, dy


def _check_column_sums(tag, dgate, dysum, a, b, dy):
    t = dy.double() * (a.double() + b.double())
    assert_within(f"{tag} dgate", dgate, t.sum(0), 1e-5, t.abs().sum(0))
    assert_within(f"{tag} dysum", dysum, dy.double().sum(0), 1e-5, dy.double().abs().sum(0))


@pytest.mark.parametrize("bdt", [torch.float32, BF16])
# one 768-thread block of 8 rows per SM, at most 148 blocks: 1184 = 148 x 8 rows is the last size with one pass of the
# grid-stride loop per block, 1185 the first with two
@pytest.mark.parametrize("rows", [1, 7, 1184, 1185, 10001, 40001])
def test_gated_residual_bwd_column_sums(rows, bdt):
    a, b, gate, dy = _gated_operands(rows, bdt, rows)
    da, db, dgate, dysum = ops.gated_residual_bwd(dy, a, b, gate, want_dysum=True)
    assert torch.equal(da, dy * (1 + gate)) and torch.equal(db, (dy * gate).to(bdt))
    _check_column_sums(f"gated_residual_bwd rows={rows} {bdt}", dgate, dysum, a, b, dy)


def test_layernorm_bwd_residual_is_dx():
    """InjectorFn.backward adds LN'(dt2) in place to the gated tail's gradient: ``residual`` and ``out`` are the same
    buffer (the tile rows of the [cls | tiles] gradient).  Bit for bit the out-of-place result."""
    rows = 10001
    g = _gen(11)
    x = torch.randn(rows, 768, generator=g, device=DEV) * 1.3 + 0.2
    w, bln = 1 + 0.1 * torch.randn(768, generator=g, device=DEV), 0.1 * torch.randn(768, generator=g, device=DEV)
    dt2, res = torch.randn(rows, 768, generator=g, device=DEV), torch.randn(rows, 768, generator=g, device=DEV)
    _, mean, rstd = ops.layernorm_fwd(x, w, bln, torch.float32)
    dx, dg, db = ops.layernorm_bwd(dt2, x, w, mean, rstd, torch.float32, residual=res, want_wgrad=True)
    buf = torch.full((rows + 1, 768), 7.0, device=DEV)
    buf[1:] = res
    dx_i, dg_i, db_i = ops.layernorm_bwd(dt2, x, w, mean, rstd, torch.float32, residual=buf[1:], want_wgrad=True,
                                         out=buf[1:])
    assert dx_i.data_ptr() == buf[1:].data_ptr() and torch.equal(dx_i, dx) and bool((buf[0] == 7.0).all())
    # dgamma / dbeta are reduced with atomics in block order: equal up to the rounding of those adds
    xhat = (x.double() - mean.double()[:, None]) * rstd.double()[:, None]
    t = dt2.double() * xhat
    assert_within("layernorm_bwd in place dgamma", dg_i, t.sum(0), 1e-5, t.abs().sum(0))
    assert_within("layernorm_bwd in place dbeta", db_i, dt2.double().sum(0), 1e-5, dt2.double().abs().sum(0))
    assert_within("layernorm_bwd dgamma in place vs out of place", dg_i, dg.double(), 1e-5, t.abs().sum(0))


def test_small_kernels_negative_control():
    """Column sums that miss the last row (a grid-stride loop that stops after its first pass at 1185 rows)."""
    a, b, gate, dy = _gated_operands(1185, torch.float32, 1185)
    _, _, dgate, dysum = ops.gated_residual_bwd(dy, a, b, gate, want_dysum=True)
    with pytest.raises(AssertionError):
        _check_column_sums("control: last row missing", dgate, dysum, a[:-1], b[:-1], dy[:-1])
