"""The float64 dilated-attention reference of tests/dilated_ref64.py (CPU): against the oracle's dilated core and its
autograd, its tile arithmetic against brute force, and the edge coverage of its geometry list."""
import pytest
import torch

from modaltune_b200 import ops
from modaltune_b200.slide_encoder import DILATED_RATIO, optimal_segment_lengths
from oracle import modaltune_oracle as O
from tests import cpu_kernels as C
from tests import dilated_ref64 as R
from tests.test_gpu_kernels import GEOMS

REF_GEOMS = GEOMS + R.EDGE_GEOMS


def _geom(N, sl):
    return ops.Geometry.get(N, sl or optimal_segment_lengths(), DILATED_RATIO)


def _qkv(geom, seed):
    g = torch.Generator().manual_seed(seed)
    qkv = torch.zeros(geom.n_alloc, 2304, dtype=torch.float64)
    qkv[:geom.n_tokens] = torch.randn(geom.n_tokens, 2304, generator=g, dtype=torch.float64) * 1.5
    return qkv


def _split(geom, qkv):
    N, H, D = geom.n_tokens, geom.heads, geom.head_dim
    return [t.reshape(N, H, D) for t in qkv[:N].split(H * D, dim=1)]


@pytest.mark.parametrize("N,sl", REF_GEOMS)
def test_fwd_ref64_matches_oracle(N, sl):
    geom = _geom(N, sl)
    qkv = _qkv(geom, N)
    _, outs, lses = O.dilated_attention_core(*_split(geom, qkv), geom.segment_lengths, geom.ratios,
                                             return_branches=True)
    o, lse, o_abs, lse_abs = R.fwd_ref64(geom, qkv)
    o_want = C._compact(geom, outs, geom.head_dim)
    lse_want = C._compact(geom, [l.unsqueeze(-1) for l in lses], 1)
    assert float((o - o_want).abs().max()) < 1e-12 and float((lse - lse_want).abs().max()) < 1e-12
    # every compact element has a writer; the absolute terms bound what they are the absolute terms of
    assert bool((lse_abs > 0).all()) and bool((o_abs >= o.abs() - 1e-12).all())


@pytest.mark.parametrize("N,sl", REF_GEOMS)
def test_bwd_ref64_matches_oracle_autograd(N, sl):
    geom = _geom(N, sl)
    qkv = _qkv(geom, N + 1)
    g = torch.Generator().manual_seed(N + 2)
    dattn = torch.zeros(geom.n_alloc, 768, dtype=torch.float64)
    dattn[:N] = torch.randn(N, 768, generator=g, dtype=torch.float64)
    q, k, v = (t.detach().requires_grad_(True) for t in _split(geom, qkv))
    out, outs, lses = O.dilated_attention_core(q, k, v, geom.segment_lengths, geom.ratios, return_branches=True)
    dq, dk, dv = torch.autograd.grad(out.reshape(N, -1), [q, k, v], dattn[:N])
    want = torch.cat([t.reshape(N, -1) for t in (dq, dk, dv)], 1)
    # the operands the kernel is handed: merged lse over the owning branches, per-branch delta = dO . o_b
    lse = torch.logsumexp(torch.stack(lses, 0).detach(), 0)
    d3 = dattn[:N].reshape(N, geom.heads, geom.head_dim)
    delta = C._compact(geom, [(d3 * ob.detach()).sum(-1, keepdim=True) for ob in outs], 1)
    got, tabs = R.bwd_ref64(geom, qkv, dattn, lse, delta)
    assert float((got - want).abs().max()) < 1e-10
    assert bool((tabs >= got.abs() - 1e-10).all())


def _brute_cells(geom, kt):
    """The same quantities by listing the positions of every slot of every (branch, segment, head)."""
    N, H = geom.n_tokens, geom.heads
    cells = []
    for sl, r in zip(geom.segment_lengths, geom.ratios):
        g = min(sl, N)
        m = -(-g // r)
        n_seg = -(-N // g)
        for s in range(n_seg):
            for h in range(H):
                off = (h * r) // H
                pos = [s * g + off + j * r for j in range(m)]
                real = [p < min(N, (s + 1) * g) for p in pos]
                tiles = [range(t, min(m, t + kt)) for t in range(0, m, kt)]
                run = [t for t in tiles if any(real[j] for j in t)]
                q_tiles = [t for t in range(0, m, 128) if any(real[j] for j in range(t, min(m, t + 128)))]
                # slots m.. of the last query tile are the first slots of segment s + 1
                past = [s * g + off + j * r for j in range(m, q_tiles[-1] + 128)] if q_tiles else []
                cells.append(dict(
                    c_real=sum(real), n_kv=len(run), n_zero_tail=sum(len(t) for t in tiles if t not in run),
                    kvalid=len(run[-1]) if run else 0, n_q=len(q_tiles),
                    q_cross=int(any(p < N for p in past) and s + 1 < n_seg)))
    return cells


SWEEP_SETS = [[16, 24, 32, 64, 128], [8, 32, 64, 96, 256], [47, 94, 188, 376, 752], [49, 98, 196, 392, 784],
              [128, 256, 512, 1024, 2048], [129, 258, 516, 1032, 2064], [1024, 5792, 32768, 185363, 1048576]]


@pytest.mark.parametrize("kt", R.KEY_TILES)
@pytest.mark.parametrize("sl", SWEEP_SETS)
def test_cell_edges_match_brute_force(sl, kt):
    Ns = list(range(1, 40)) + list(range(40, 700, 7)) + [1023, 1024, 1025, 2049, 5793]
    for N in Ns:
        if any(-(-N // min(s, N)) > 1 and min(s, N) % r for s, r in zip(sl, DILATED_RATIO)):
            continue   # several segments whose length the dilation does not divide: rejected by the library
        geom = ops.Geometry(N, sl, DILATED_RATIO)
        got = R.cell_edges(geom, kt)
        want = _brute_cells(geom, kt)
        assert len(got) == len(want)
        for a, b in zip(got, want):
            assert {k: a[k] for k in b} == b, (N, sl, kt, a, b)


@pytest.mark.parametrize("kt", R.KEY_TILES)
def test_edge_geometries_cover_every_condition(kt):
    hit = set()
    for N, sl in R.EDGE_GEOMS:
        hit |= R.edges_hit(_geom(N, sl), kt)
    missing = set(R.EDGE_CONDITIONS) | set(R.GEOMETRY_CONDITIONS)
    missing -= hit
    assert not missing, f"kt={kt}: no geometry of EDGE_GEOMS reaches {sorted(missing)}"
