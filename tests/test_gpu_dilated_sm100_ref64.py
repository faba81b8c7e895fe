"""The tcgen05 dilated-attention kernels (forward impls 1 / 3, backward impls 1 / 2 / 4) held per element to the float64
reference of tests/dilated_ref64.py, at the tile edges of tests/dilated_ref64.EDGE_GEOMS and at bench sizes, in three
input regimes; the work counter of the persistent backward across geometries and around its ring; and negative
controls: deliberately wrong references that the same checks must reject.

Error model (bf16 operands, fp32 accumulation, dilated_sm100.cu):
- forward o: P is rounded to bf16 (relative 2^-9) before P V, so |o - o_ref| <= 2^-9 sum_j P_ij |v_jd| plus fp32
  accumulation; the bf16 store of o adds 2^-9 |o|.  Bound: 2^-8 sum_j P_ij |v_jd| + 2^-8 |o_ref|.
- forward lse = m scale + log(l): l is an fp32 sum of unrounded ex2 values (relative error ~1e-6 at a few thousand
  terms), log and the product by scale are fp32; the scores themselves carry the fp32 rounding of the three K = 16
  MMA steps, < 2^-20 sum_d |q_id k_jd| per score.  Bound: 1e-5 (1 + |lse_ref|) + 2^-20 scale max_j sum_d |q_id k_jd|.
- backward: P (for dV) and dS = P (dO V^T - delta) (for dQ, dK) are rounded to bf16 before their MMAs, 2^-9 of the
  absolute terms each, with fp32 accumulation across key and query tiles.  Bound: 2^-7 of T_dq / T_dk / T_dv.
"""
import pytest
import torch

from modaltune_b200 import _lib, ops
from modaltune_b200.slide_encoder import DILATED_RATIO, optimal_segment_lengths
from tests import dilated_ref64 as R

pytestmark = pytest.mark.gpu
DEV = "cuda"

FWD_IMPLS = (1, 3)         # 128-key and 48-key (default) score tiles
BWD_IMPLS = (1, 2, 4)      # one CTA per key tile, persistent (default), deterministic
O_BOUND = 2.0 ** -8
LSE_REL, LSE_ABS = 1e-5, 2.0 ** -20
BWD_BOUND = 2.0 ** -7
GEOMS = R.EDGE_GEOMS + [(5793, None), (10001, None), (32769, None), (40001, None)]
REGIMES = ("randn", "flat", "rising")


def _geom(N, sl):
    return ops.Geometry.get(N, sl or optimal_segment_lengths(), DILATED_RATIO)


def _qkv(geom, regime, seed):
    """randn x 1.5; flat: x 0.05, so zero keys weigh as much as real ones; rising: key magnitudes growing 9x along
    the sequence with the sign flipped every 128 positions, so row maxima jump by more than the lazy-rescale threshold."""
    N = geom.n_tokens
    g = torch.Generator().manual_seed(seed)
    qkv = torch.zeros(geom.n_alloc, 2304)
    qkv[:N] = torch.randn(N, 2304, generator=g)
    if regime == "randn":
        qkv[:N] *= 1.5
    elif regime == "flat":
        qkv[:N] *= 0.05
    else:
        ramp = (1.0 + 8.0 * torch.arange(N) / N).unsqueeze(1)
        sign = torch.where(torch.arange(N) % 256 < 128, 1.0, -1.0).unsqueeze(1)
        qkv[:N, 768:1536] *= ramp * sign
    return qkv.to(torch.bfloat16).to(DEV)


def _fwd(geom, qkv, impl):
    """mt_dilated_attn_fwd into NaN-filled outputs: every compact element must be written by exactly one CTA."""
    o = torch.full((geom.o_elems,), float("nan"), device=DEV, dtype=torch.bfloat16)
    lse = torch.full((geom.lse_elems,), float("nan"), device=DEV, dtype=torch.float32)
    rc = _lib.load().mt_dilated_attn_fwd(geom.ref(), ops._p(qkv), qkv.stride(0), qkv.shape[0], ops._dt(qkv), ops._p(o),
                                         ops._p(lse), impl, ops._stream())
    assert rc == 0, _lib.last_error()
    return o, lse


def _ratio(err, bound):
    return float(torch.where(err == 0, torch.zeros_like(err), err / bound).max())


def fwd_ratios(o, lse, ref):
    """Largest err / bound of o (2^-8 (sum_j P|v| + |o_ref|)) and of lse (1e-5 (1 + |lse|) + 2^-20 scale max sum|qk|)."""
    o_ref, lse_ref, o_abs, lse_abs = ref
    return {"o": _ratio((o.double() - o_ref).abs(), O_BOUND * (o_abs + o_ref.abs())),
            "lse": _ratio((lse.double() - lse_ref).abs(), LSE_REL * (1 + lse_ref.abs()) + LSE_ABS * lse_abs)}


def check_fwd(o, lse, ref, what=""):
    assert bool(torch.isfinite(o.float()).all()) and bool(torch.isfinite(lse).all()), (what, "unwritten or non-finite")
    e = fwd_ratios(o, lse, ref)
    print(f"ref64 fwd {what}: " + " ".join(f"{k} {v:.3g}" for k, v in e.items()) + " (of the bound)")
    assert max(e.values()) <= 1.0, (what, e)
    return e


def bwd_ratios(dqkv, ref, tabs):
    """Largest err / bound of dq, dk, dv, each bound 2^-7 of its sum of absolute terms."""
    return {name: _ratio((dqkv[:, cols].double() - ref[:, cols]).abs(), BWD_BOUND * tabs[:, cols])
            for name, cols in (("dq", slice(0, 768)), ("dk", slice(768, 1536)), ("dv", slice(1536, 2304)))}


def check_bwd(dqkv, ref, tabs, what=""):
    assert bool(torch.isfinite(dqkv).all()), what
    e = bwd_ratios(dqkv, ref, tabs)
    print(f"ref64 bwd {what}: " + " ".join(f"{k} {v:.3g}" for k, v in e.items()) + " (of the bound)")
    assert max(e.values()) <= 1.0, (what, e)
    return e


def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max())


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("N,sl", GEOMS)
def test_forward_per_element(N, sl, regime):
    geom = _geom(N, sl)
    qkv = _qkv(geom, regime, N + 1)
    ref = R.fwd_ref64(geom, qkv)
    for impl in FWD_IMPLS:
        o, lse = _fwd(geom, qkv, impl)
        torch.cuda.synchronize()
        check_fwd(o, lse, ref, f"impl {impl} N={N} {regime}")


def _bwd_inputs(geom, qkv, seed):
    """dO, merged lse and per-branch delta as the training step makes them: forward impl 3, merge + LayerNorm."""
    g = torch.Generator().manual_seed(seed)
    gamma = (1 + 0.1 * torch.randn(768, generator=g)).to(DEV)
    beta = (0.1 * torch.randn(768, generator=g)).to(DEV)
    dy = torch.randn(geom.n_tokens, 768, generator=g).to(DEV)
    o, l = ops.dilated_attn_fwd(geom, qkv, 3)
    _, _, lse, m, r = ops.dilated_merge_ln_fwd(geom, o, l, gamma, beta)
    dattn, delta = ops.dilated_merge_ln_bwd(geom, dy, o, l, gamma, m, r)
    return dattn, lse, delta, l


def _bwd(geom, qkv, dattn, lse, delta, impl):
    assert ops.dilated_bwd_impl(impl) == impl
    return ops.dilated_attn_bwd(geom, qkv, dattn, lse, delta, impl)


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("N,sl", GEOMS)
def test_backward_per_element(N, sl, regime):
    geom = _geom(N, sl)
    qkv = _qkv(geom, regime, N + 2)
    dattn, lse, delta, _ = _bwd_inputs(geom, qkv, N + 3)
    ref, tabs = R.bwd_ref64(geom, qkv, dattn, lse, delta)
    for impl in BWD_IMPLS:
        d = _bwd(geom, qkv, dattn, lse, delta, impl)
        torch.cuda.synchronize()
        check_bwd(d, ref, tabs, f"impl {impl} N={N} {regime}")


def test_bwd_impl2_back_to_back_geometries():
    """Persistent backward launches on a large, a small and a large geometry in a row, each with its own work counter."""
    runs = []
    for N, sl in ((10001, None), (60, [47, 94, 188, 376, 752]), (5793, None)):
        geom = _geom(N, sl)
        qkv = _qkv(geom, "randn", N + 4)
        runs.append((geom, qkv) + _bwd_inputs(geom, qkv, N + 5)[:3])
    outs = [_bwd(geom, qkv, dattn, lse, delta, 2) for geom, qkv, dattn, lse, delta in runs]
    torch.cuda.synchronize()
    for (geom, qkv, dattn, lse, delta), d in zip(runs, outs):
        check_bwd(d, *R.bwd_ref64(geom, qkv, dattn, lse, delta), f"impl 2 back to back N={geom.n_tokens}")


def test_bwd_impl2_counter_ring_wraps():
    """300 launches in a row take every pair of the 256-entry counter ring at least once; a pair that was not re-armed
    would hand its next launch no (or too few) work items and leave rows of the memset output at zero."""
    geom = _geom(193, [49, 98, 196, 392, 784])
    qkv = _qkv(geom, "randn", 6)
    dattn, lse, delta, _ = _bwd_inputs(geom, qkv, 7)
    ref, tabs = R.bwd_ref64(geom, qkv, dattn, lse, delta)
    for i in range(300):
        d = _bwd(geom, qkv, dattn, lse, delta, 2)
        assert bool(torch.isfinite(d[:, :768]).all()), i
        if i in (0, 256, 299):
            check_bwd(d, ref, tabs, f"impl 2 call {i + 1} of 300")
        else:
            assert max(bwd_ratios(d, ref, tabs).values()) <= 1.0, i


# ---------------------------------------------------------------------------------------------------------------------
# negative controls: a wrong reference must fail the same checks (and the old global bars are reported next to it)
# ---------------------------------------------------------------------------------------------------------------------
def _cell_lse_index(geom, cell):
    """Compact lse indices of the real positions of one (branch, segment, head) cell."""
    _, _, _, _, hpb, slot_off = R._branches(geom)[cell["b"]]
    pos = cell["s"] * cell["g"] + cell["off"] + cell["r"] * torch.arange(cell["c_real"])
    return slot_off + pos * hpb + (cell["h"] - cell["off"] * hpb)


def _old_fwd_bars(o, lse, ref):
    return _rel(o, ref[0]) < 3e-2 and float((lse.double() - ref[1]).abs().max()) < 2e-2


def _old_bwd_bars(d, ref):
    ok = True
    for cols in (slice(0, 768), slice(768, 1536), slice(1536, 2304)):
        a, b = d[:, cols].double().flatten(), ref[:, cols].flatten()
        ok &= _rel(a, b) < 3e-2 and float(torch.nn.functional.cosine_similarity(a, b, dim=0)) > 0.9995
    return ok


def _fwd_control(N, sl, regime, wrong, which):
    """Forward impl 3 passes against the right reference and fails on ``which`` against the wrong one."""
    geom = _geom(N, sl)
    qkv = _qkv(geom, regime, N + 1)
    o, lse = _fwd(geom, qkv, 3)
    torch.cuda.synchronize()
    check_fwd(o, lse, R.fwd_ref64(geom, qkv), "control baseline")
    bad = wrong(geom, qkv)
    print(f"control: {fwd_ratios(o, lse, bad)} of the bound; old bars accept it: {_old_fwd_bars(o, lse, bad)}")
    with pytest.raises(AssertionError):
        check_fwd(o, lse, bad, "wrong reference")
    assert fwd_ratios(o, lse, bad)[which] > 1.0


def test_control_zero_tail_one_key_short():
    """Flat scores at N = 513: the cells of one real slot of 512 add 464 zero keys in closed form; one fewer moves
    lse by -log(1 - 1/l) ~ 2e-3."""
    def wrong(geom, qkv):
        o, lse, o_abs, lse_abs = (t.clone() for t in R.fwd_ref64(geom, qkv))
        for c in R.cell_edges(geom, 48):
            if c["c_real"] > 0 and c["n_zero_tail"] > 0:
                i = _cell_lse_index(geom, c).to(DEV)
                l = lse[i].exp()
                lse[i] = torch.log(l - 1)       # a zero key contributes exp(0) = 1 to l and nothing to o l
                oi = (i[:, None] * 48 + torch.arange(48, device=DEV)).reshape(-1)
                o[oi] *= (l / (l - 1)).repeat_interleave(48)
        return o, lse, o_abs, lse_abs
    _fwd_control(513, [512, 1024, 2048, 4096, 8192], "flat", wrong, "lse")


def test_control_last_slot_dropped():
    _fwd_control(129, [128, 256, 512, 1024, 2048], "randn", lambda geom, qkv: R.fwd_ref64(geom, qkv, n_keys=lambda m: m - 1),
                 "o")


def test_control_next_segment_slot_included():
    _fwd_control(129, [128, 256, 512, 1024, 2048], "randn", lambda geom, qkv: R.fwd_ref64(geom, qkv, n_keys=lambda m: m + 1),
                 "o")


def _bwd_control(N, sl, impl, wrong, which):
    geom = _geom(N, sl)
    qkv = _qkv(geom, "randn", N + 2)
    dattn, lse, delta, lse_br = _bwd_inputs(geom, qkv, N + 3)
    d = _bwd(geom, qkv, dattn, lse, delta, impl)
    torch.cuda.synchronize()
    check_bwd(d, *R.bwd_ref64(geom, qkv, dattn, lse, delta), "control baseline")
    bad, tabs = wrong(geom, qkv, dattn, lse, delta, lse_br)
    print(f"control: {bwd_ratios(d, bad, tabs)} of the bound; old bars accept it: {_old_bwd_bars(d, bad)}")
    with pytest.raises(AssertionError):
        check_bwd(d, bad, tabs, "wrong reference")
    assert all(bwd_ratios(d, bad, tabs)[w] > 1.0 for w in which)


def test_control_neighbouring_head_delta():
    """Branch 0 (16 head slots per position) reads the delta of head slot h + 1: dq of every row moves."""
    def wrong(geom, qkv, dattn, lse, delta, lse_br):
        N = geom.n_tokens
        bad = delta.clone()
        bad[:N * 16] = delta[:N * 16].view(N, 16).roll(1, dims=1).reshape(-1)
        return R.bwd_ref64(geom, qkv, dattn, lse, bad)
    _bwd_control(257, [129, 258, 516, 1032, 2064], 2, wrong, ["dq"])


def test_control_partial_query_tile_row_left_out():
    """N = 257, segment 129: the second query tile of segment 0 holds the single slot 128; leaving that row out of
    dk / dv moves the keys it attends to."""
    def wrong(geom, qkv, dattn, lse, delta, lse_br):
        return R.bwd_ref64(geom, qkv, dattn, lse, delta, kv_skip_row=128)
    _bwd_control(257, [129, 258, 516, 1032, 2064], 2, wrong, ["dk", "dv"])


def test_control_branch_lse_instead_of_merged():
    """P formed with the lse of branch 0 alone instead of the merged lse."""
    def wrong(geom, qkv, dattn, lse, delta, lse_br):
        return R.bwd_ref64(geom, qkv, dattn, lse_br[:geom.n_tokens * 16].view(geom.n_tokens, 16), delta)
    _bwd_control(255, [192, 384, 768, 1536, 3072], 1, wrong, ["dq", "dk", "dv"])
