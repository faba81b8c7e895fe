"""Float64 reference of the dilated-attention core and the tile arithmetic of the tcgen05 kernels (helper module).

``cell_edges`` restates, per (branch, segment, head), the integer arithmetic with which the tcgen05 kernels of
``modaltune_b200/csrc/dilated_sm100.cu`` skip padding and mask the segment boundary.  ``fwd_ref64`` / ``bwd_ref64`` give the
exact results of the kernels' own operands in the kernels' compact layouts, together with the sums of absolute terms
that per-element error bounds are stated in.  Everything runs on the device of the inputs (CPU or CUDA), batched over
the segments and heads of a branch.
"""
from __future__ import annotations

from typing import Dict, List

import torch

QUERY_TILE = 128          # query slots per CTA in every tcgen05 kernel
KEY_TILES = (48, 128)     # key slots per score tile: 48 (forward impl 3, dQ of backward impl 4), 128 (the others)
CHUNK_ELEMS = 1 << 27     # score-matrix elements per batch of cells (1 GiB of float64 per temporary)


def _branches(geom):
    """Per branch: (r, g, m, n_seg, hpb, offset in o_br / lse_br in units of one head slot)."""
    N, H = geom.n_tokens, geom.heads
    out, slot_off = [], 0
    for sl, r in zip(geom.segment_lengths, geom.ratios):
        g = min(sl, N)
        out.append((r, g, -(-g // r), -(-N // g), H // r, slot_off))
        slot_off += N * (H // r)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# tile arithmetic
# ---------------------------------------------------------------------------------------------------------------------
def cell_edges(geom, kt: int) -> List[Dict[str, int]]:
    """One dict per (branch, segment, head) with key tiles of ``kt`` slots, in the kernels' integer arithmetic:

    ``m`` slots per segment, residue ``off``, ``c_real`` slots at a position < N, ``n_kv`` key tiles computed (the others
    are all zero keys), ``n_zero_tail`` zero keys added in closed form, ``kvalid`` slots of the last computed key tile
    that are not masked (a tile masks when kvalid < kt), ``n_q`` 128-slot query tiles that run, and ``q_cross``: the last
    query tile reaches slots past ``m`` that are real positions of the following segment.
    """
    N, H = geom.n_tokens, geom.heads
    cells = []
    for b, (r, g, m, n_seg, _, _) in enumerate(_branches(geom)):
        for s in range(n_seg):
            seg_end = min(N, (s + 1) * g)
            for h in range(H):
                off = (h * r) // H
                seg_lo = s * g + off
                c_real = (seg_end - seg_lo + r - 1) // r if seg_end > seg_lo else 0
                n_kv = min(-(-m // kt), -(-c_real // kt))
                n_q = -(-c_real // QUERY_TILE)
                cells.append(dict(
                    b=b, s=s, h=h, r=r, g=g, m=m, off=off, c_real=c_real, n_kv=n_kv,
                    n_zero_tail=max(0, m - n_kv * kt) if c_real > 0 else m,
                    kvalid=min(kt, m - (n_kv - 1) * kt) if n_kv > 0 else 0,
                    n_q=n_q,
                    q_cross=int(c_real > 0 and n_q * QUERY_TILE > m and (s + 1) * g + off < N),
                    next_real=int((s + 1) * g + off < N)))
    return cells


# the edge conditions a geometry list has to reach, for a key tile of kt slots
EDGE_CONDITIONS = {
    "c_real == 0": lambda c, kt: c["c_real"] == 0,
    "partial segment, c_real % kt == 0": lambda c, kt: 0 < c["c_real"] < c["m"] and c["c_real"] % kt == 0,
    "partial segment, c_real % kt == 1": lambda c, kt: 0 < c["c_real"] < c["m"] and c["c_real"] % kt == 1,
    "partial segment, c_real % kt == kt-1": lambda c, kt: 0 < c["c_real"] < c["m"] and c["c_real"] % kt == kt - 1,
    "n_zero_tail == 0, c_real < m": lambda c, kt: 0 < c["c_real"] < c["m"] and c["n_zero_tail"] == 0,
    "n_zero_tail in 1..kt-1": lambda c, kt: c["c_real"] > 0 and 1 <= c["n_zero_tail"] <= kt - 1,
    "n_zero_tail >= 2 kt": lambda c, kt: c["c_real"] > 0 and c["n_zero_tail"] >= 2 * kt,
    "m % kt == 0, next segment real": lambda c, kt: c["next_real"] and c["m"] % kt == 0,
    "m % kt == 1, next segment real": lambda c, kt: c["next_real"] and c["m"] % kt == 1,
    "m % kt == kt-1, next segment real": lambda c, kt: c["next_real"] and c["m"] % kt == kt - 1,
    "query tile crosses into the next segment": lambda c, kt: c["q_cross"] == 1,
}
GEOMETRY_CONDITIONS = {
    "g > N": lambda geom: any(sl > geom.n_tokens for sl in geom.segment_lengths),
    "N < 16": lambda geom: geom.n_tokens < 16,
}


# (N, segment lengths) with the dilations (1, 2, 4, 8, 16): together they reach every condition above for both key
# tiles (tests/test_dilated_ref64.py checks it).  Chosen by a greedy scan over N < 3000 and segment-length sets
# a * (1, 2, 4, 8, 16), for the least float64 work per newly reached condition.
EDGE_GEOMS = [
    (11, [8, 32, 64, 96, 256]),             # N < 16, g > N, (segment, head) cells without a real position
    (60, [47, 94, 188, 376, 752]),          # m = 47 = 48 - 1 with the next segment real
    (128, [127, 254, 508, 1016, 2032]),     # m = 127 = 128 - 1 with the next segment real; a one-position segment
    (129, [128, 256, 512, 1024, 2048]),     # m = 128 with the next segment real; a one-position segment
    (193, [49, 98, 196, 392, 784]),         # m = 49 = 48 + 1; partial segments of 46, 47 and 48 real slots
    (255, [192, 384, 768, 1536, 3072]),     # m = 192 = 4 x 48; 63 real slots of 192: 96 / 64 zero keys in closed form
    (257, [129, 258, 516, 1032, 2064]),     # m = 129 = 128 + 1; 128 real slots of 129: one zero key in closed form
    (513, [512, 1024, 2048, 4096, 8192]),   # one real slot of 512: 464 / 384 zero keys in closed form
]


def edges_hit(geom, kt: int) -> set:
    hit = {name for name, f in GEOMETRY_CONDITIONS.items() if f(geom)}
    for c in cell_edges(geom, kt):
        hit |= {name for name, f in EDGE_CONDITIONS.items() if f(c, kt)}
    return hit


# ---------------------------------------------------------------------------------------------------------------------
# float64 references
# ---------------------------------------------------------------------------------------------------------------------
def _gather(geom, r, g, m, n_seg, hpb, x64, cols0):
    """Per cell (segment, residue, head slot): the m slots of columns [cols0 + h*D, +D) as [n_seg*r*hpb, m, D], zero for
    positions >= N; also the positions [n_seg, r, m] and their mask pos < N."""
    N, D = geom.n_tokens, geom.head_dim
    dev = x64.device
    pos = (torch.arange(n_seg, device=dev)[:, None, None] * g + torch.arange(r, device=dev)[None, :, None]
           + r * torch.arange(m, device=dev)[None, None, :])                 # [n_seg, r, m]
    real = pos < N
    pc = torch.where(real, pos, torch.full_like(pos, N))                      # row N of the padded copy is zero
    heads = torch.arange(r, device=dev)[:, None] * hpb + torch.arange(hpb, device=dev)[None, :]   # [r, hpb]
    cols = cols0 + heads[:, :, None] * D + torch.arange(D, device=dev)        # [r, hpb, D]
    t = x64[pc[:, :, None, :, None], cols[None, :, :, None, :]]              # [n_seg, r, hpb, m, D]
    return t.reshape(n_seg * r * hpb, m, D), pos, real


def _padded(t, N):
    return torch.cat([t[:N].double(), torch.zeros(1, t.shape[1], dtype=torch.float64, device=t.device)], 0)


def _chunks(n_cells, m):
    step = max(1, CHUNK_ELEMS // (m * m))
    return [(i, min(n_cells, i + step)) for i in range(0, n_cells, step)]


def _slot_index(pos, real, hpb, slot_off):
    """Compact index (lse layout: [N][hpb] per branch) of every (cell, slot), -1 for positions >= N."""
    n_seg, r, m = pos.shape
    idx = slot_off + pos[:, :, None, :] * hpb + torch.arange(hpb, device=pos.device)[None, None, :, None]
    return torch.where(real[:, :, None, :], idx, torch.full_like(idx, -1)).reshape(n_seg * r * hpb, m)


def fwd_ref64(geom, qkv, n_keys=None):
    """Per-branch output and log-sum-exp of the dilated core in float64, from the bf16 / fp32 qkv the kernel reads.

    Returns ``(o, lse, o_abs, lse_abs)`` in the compact layouts of ``mt_dilated_attn_fwd`` (``o_elems`` / ``lse_elems``):
    ``o_abs = sum_j P_ij |v_jd|`` and ``lse_abs = scale * max_j sum_d |q_id k_jd|``.  Keys at positions >= N are zero keys
    (score 0, value 0, counted in the denominator); slots past the segment's m do not exist.  ``n_keys(m)``, for
    negative controls only, replaces the m key slots of every segment by that many (m - 1 drops the last slot, m + 1
    adds the first slot of the next segment).
    """
    N, H, D = geom.n_tokens, geom.heads, geom.head_dim
    E = H * D
    sc = D ** -0.5
    dev = qkv.device
    x = _padded(qkv, N)
    o = torch.zeros(geom.o_elems, dtype=torch.float64, device=dev)
    o_abs = torch.zeros_like(o)
    lse = torch.zeros(geom.lse_elems, dtype=torch.float64, device=dev)
    lse_abs = torch.zeros_like(lse)
    for r, g, m, n_seg, hpb, slot_off in _branches(geom):
        mk = n_keys(m) if n_keys is not None else m
        q, pos, real = _gather(geom, r, g, m, n_seg, hpb, x, 0)
        k, _, _ = _gather(geom, r, g, mk, n_seg, hpb, x, E)
        v, _, _ = _gather(geom, r, g, mk, n_seg, hpb, x, 2 * E)
        idx = _slot_index(pos, real, hpb, slot_off)
        for a, e in _chunks(q.shape[0], max(m, mk)):
            s = q[a:e] @ k[a:e].transpose(1, 2) * sc
            l = torch.logsumexp(s, -1)
            p = torch.exp(s - l[..., None])
            ob, tb = p @ v[a:e], p @ v[a:e].abs()
            la = (q[a:e].abs() @ k[a:e].abs().transpose(1, 2)).amax(-1) * sc
            i = idx[a:e]
            ok = i >= 0
            lse[i[ok]], lse_abs[i[ok]] = l[ok], la[ok]
            oi = (i[ok][:, None] * D + torch.arange(D, device=dev)).reshape(-1)
            o[oi], o_abs[oi] = ob[ok].reshape(-1), tb[ok].reshape(-1)
            del s, p
    return o, lse, o_abs, lse_abs


def bwd_ref64(geom, qkv, dattn, lse, delta_br, kv_skip_row=None):
    """dq | dk | dv [N, 3E] in float64 from the operands ``mt_dilated_attn_bwd`` takes: the merged lse [N, H] and the
    per-branch delta (compact layout).  Per cell P = exp(S - lse), dS = P (dO V^T - delta_b), dq = sc dS K,
    dk = sc dS^T Q, dv = P^T dO.  Also returns the sums of absolute terms [N, 3E], added over branches:
    T_dq = sc (P (|dO| |V|^T + |delta|)) |K|, T_dk = sc (P (|dO| |V|^T + |delta|))^T |Q|, T_dv = P^T |dO|.
    ``kv_skip_row``, for negative controls only: a position whose query row is left out of dk and dv.
    """
    N, H, D = geom.n_tokens, geom.heads, geom.head_dim
    E = H * D
    sc = D ** -0.5
    dev = qkv.device
    x, do = _padded(qkv, N), _padded(dattn, N)
    lse_p = _padded(lse.reshape(N, H), N)
    dlt = torch.cat([delta_br.double(), torch.zeros(1, dtype=torch.float64, device=dev)])
    out = torch.zeros(N + 1, 3 * E, dtype=torch.float64, device=dev)      # row N collects the padding slots
    tabs = torch.zeros_like(out)
    for r, g, m, n_seg, hpb, slot_off in _branches(geom):
        q, pos, real = _gather(geom, r, g, m, n_seg, hpb, x, 0)
        k, _, _ = _gather(geom, r, g, m, n_seg, hpb, x, E)
        v, _, _ = _gather(geom, r, g, m, n_seg, hpb, x, 2 * E)
        dO, _, _ = _gather(geom, r, g, m, n_seg, hpb, do, 0)
        # merged lse and delta of every (cell, slot): head h = residue * hpb + head slot of the cell
        pc = torch.where(real, pos, torch.full_like(pos, N))
        heads = torch.arange(r, device=dev)[:, None] * hpb + torch.arange(hpb, device=dev)[None, :]
        L = lse_p[pc[:, :, None, :], heads[None, :, :, None]].reshape(-1, m)
        di = _slot_index(pos, real, hpb, slot_off)
        dl = dlt[torch.where(di >= 0, di, torch.full_like(di, dlt.numel() - 1))]
        rows = pc[:, :, None, :].expand(n_seg, r, hpb, m).reshape(-1, m)
        cols = (heads[None, :, :, None] * D).expand(n_seg, r, hpb, 1).reshape(-1, 1) + torch.arange(D, device=dev)
        mask = real[:, :, None, :].expand(n_seg, r, hpb, m).reshape(-1, m).double()
        for a, e in _chunks(q.shape[0], m):
            p = torch.exp(q[a:e] @ k[a:e].transpose(1, 2) * sc - L[a:e, :, None]) * mask[a:e, :, None]
            ds = p * (dO[a:e] @ v[a:e].transpose(1, 2) - dl[a:e, :, None])
            ta = p * (dO[a:e].abs() @ v[a:e].abs().transpose(1, 2) + dl[a:e, :, None].abs())
            dq, tq = ds @ k[a:e] * sc, ta @ k[a:e].abs() * sc
            if kv_skip_row is not None:
                keep = (rows[a:e] != kv_skip_row).double()[:, :, None]
                p, ds, ta = p * keep, ds * keep, ta * keep
            for j, (val, tval) in enumerate(((dq, tq),
                                             (ds.transpose(1, 2) @ q[a:e] * sc, ta.transpose(1, 2) @ q[a:e].abs() * sc),
                                             (p.transpose(1, 2) @ dO[a:e], p.transpose(1, 2) @ dO[a:e].abs()))):
                ri = rows[a:e, :, None].expand(-1, -1, D)
                ci = (cols[a:e, None, :] + j * E).expand(-1, m, -1)
                out.index_put_((ri.reshape(-1), ci.reshape(-1)), val.reshape(-1), accumulate=True)
                tabs.index_put_((ri.reshape(-1), ci.reshape(-1)), tval.reshape(-1), accumulate=True)
            del p, ds, ta
    return out[:N], tabs[:N]
