"""Thin Python side of the C ABI: tensor -> pointer marshalling and the ``torch.autograd.Function``s of the hot path.

Every function here launches hand-written sm_100a kernels from ``libmodaltune_b200.so`` on the current CUDA stream;
dense projections between them are plain cuBLAS GEMMs (``torch.nn.functional.linear`` / ``torch.matmul``).  Nothing in
this module has a CPU implementation: tensors must live on a CUDA device.

Reference functions replaced (paths relative to the reference root, ``TS/`` =
``models/prov_gigapath/gigapath/torchscale/``): ``TS/architecture/encoder.py:121-175`` (EncoderLayer.forward),
``TS/component/dilated_attention.py:82-262``, ``TS/component/multihead_attention.py:109-119``,
``TS/component/feedforward_network.py:132-143``, ``models/vitadapter/adapter_modules.py:210-234, 321-369``.
"""
from __future__ import annotations

import ctypes
import math
import weakref
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import MT_BF16, MT_F32, DilatedGeometry

HEADS = 16
HEAD_DIM = 48
EMBED = 768
LN_EPS = 1e-5

# kernel-launch counter (bench.py reports it as `gpu_launches`); incremented once per C-ABI launch call
launch_count = 0
# optional per-kernel CUDA-event timing (bench.py's roofline leg): name -> [(start_event, stop_event), ...]
kernel_events = None


class _timed:
    """Record CUDA events on the launching stream around one kernel when ``kernel_events`` is a dict."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if kernel_events is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.stop = torch.cuda.Event(enable_timing=True)
            self.start.record()
        return self

    def __exit__(self, *exc):
        if kernel_events is not None:
            self.stop.record()
            kernel_events.setdefault(self.name, []).append((self.start, self.stop))
        return False


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return MT_F32
    if t.dtype == torch.bfloat16:
        return MT_BF16
    raise TypeError(f"unsupported dtype {t.dtype} (float32 / bfloat16 only)")


def _p(t: Optional[torch.Tensor]):
    if t is None:
        return None
    assert t.is_cuda, "modaltune_b200 kernels need CUDA tensors (there is no CPU path)"
    assert t.is_contiguous(), "modaltune_b200 kernels need contiguous tensors"
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check(rc: int, what: str, launches: int = 1) -> None:
    global launch_count
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {_lib.last_error()}")
    launch_count += launches


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t if t.dtype == torch.float32 else t.float()


def _deterministic() -> bool:
    from . import config
    return config.deterministic()


def _colreduce_workspace(device, cols: int) -> torch.Tensor:
    """Block partials of a deterministic column reduction (``mt_*_ws``); under graph capture from the graph's pool."""
    return torch.empty(int(_lib.load().mt_colreduce_workspace_floats(cols)), device=device, dtype=torch.float32)


# ---------------------------------------------------------------------------------------------------------------------
# dilated-attention geometry
# ---------------------------------------------------------------------------------------------------------------------
class Geometry:
    """Host mirror of ``mt_dilated_geometry`` + the compact per-branch buffer sizes (include/modaltune_b200.h)."""

    _cache: Dict[tuple, "Geometry"] = {}

    def __init__(self, n_tokens: int, segment_lengths: Sequence[int], ratios: Sequence[int], heads: int = HEADS,
                 head_dim: int = HEAD_DIM):
        assert len(segment_lengths) == len(ratios) <= _lib.MT_MAX_BRANCHES
        self.n_tokens, self.heads, self.head_dim = int(n_tokens), heads, head_dim
        self.segment_lengths = [int(s) for s in segment_lengths]
        self.ratios = [int(r) for r in ratios]
        g = DilatedGeometry()
        g.n_tokens, g.n_heads, g.head_dim, g.n_branches = self.n_tokens, heads, head_dim, len(ratios)
        self.o_elems = 0
        self.lse_elems = 0
        self.flops_fwd = 0.0  # algorithmic: 4 * d * sum c^2 over real positions only (SURVEY.md §8d)
        for b, (sl, r) in enumerate(zip(self.segment_lengths, self.ratios)):
            g.seg_len[b] = min(sl, 2**31 - 1)
            g.ratio[b] = r
            assert heads % r == 0, "dilation must divide the head count"
            self.o_elems += self.n_tokens * (heads // r) * head_dim
            self.lse_elems += self.n_tokens * (heads // r)
            gl = min(sl, self.n_tokens)
            n_seg = -(-self.n_tokens // gl)
            for s in range(n_seg):
                lo, hi = s * gl, min(self.n_tokens, (s + 1) * gl)
                for h in range(heads):
                    off = (h * r) // heads
                    c = max(0, -(-(hi - lo - off) // r))
                    self.flops_fwd += 4.0 * head_dim * c * c
        self.c_struct = g
        self.n_alloc = -(-self.n_tokens // 128) * 128  # qkv rows incl. the zero tail the TMA path reads

    @classmethod
    def get(cls, n_tokens: int, segment_lengths: Sequence[int], ratios: Sequence[int]) -> "Geometry":
        key = (int(n_tokens), tuple(int(s) for s in segment_lengths), tuple(int(r) for r in ratios))
        if key not in cls._cache:
            cls._cache[key] = Geometry(*key)
        return cls._cache[key]

    def ref(self):
        return ctypes.byref(self.c_struct)


# ---------------------------------------------------------------------------------------------------------------------
# raw kernel wrappers (no autograd)
# ---------------------------------------------------------------------------------------------------------------------
def layernorm_fwd(x, gamma, beta, out_dtype, add=None, eps: float = LN_EPS, want_stats: bool = True):
    rows, cols = x.shape
    y = torch.empty((rows, cols), device=x.device, dtype=out_dtype)
    mean = torch.empty(rows, device=x.device, dtype=torch.float32) if want_stats else None
    rstd = torch.empty(rows, device=x.device, dtype=torch.float32) if want_stats else None
    add_rows = add.shape[0] if add is not None else 1
    rc = _lib.load().mt_layernorm_fwd(_p(x), _dt(x), _p(gamma), _p(beta), _p(add), _dt(add) if add is not None else 0,
                                      add_rows, _p(y), _dt(y), _p(mean), _p(rstd), rows, cols, eps, _stream())
    _check(rc, "mt_layernorm_fwd")
    return y, mean, rstd


def layernorm_bwd(dy, x, gamma, mean, rstd, dx_dtype, residual=None, want_wgrad: bool = False, out=None,
                  bf16_twin: bool = False):
    """``bf16_twin``: also write dx rounded to bf16 in the same pass (kept as ``dx._mt_bf16``): the next GEMM of the
    backward chain takes it instead of running a separate cast over the tensor."""
    rows, cols = x.shape
    dx = out if out is not None else torch.empty((rows, cols), device=x.device, dtype=dx_dtype)
    twin = torch.empty((rows, cols), device=x.device, dtype=torch.bfloat16) if bf16_twin else None
    dgamma = dbeta = None
    lib = _lib.load()
    args = (_p(dy), _dt(dy), _p(x), _dt(x), _p(gamma), _p(mean), _p(rstd), _p(residual),
            _dt(residual) if residual is not None else 0, _p(dx), _dt(dx), _p(twin))
    if want_wgrad and _deterministic():
        dgb = torch.empty((2, cols), device=x.device, dtype=torch.float32)   # written, not accumulated
        dgamma, dbeta = dgb[0], dgb[1]
        ws = _colreduce_workspace(x.device, cols)
        rc = lib.mt_layernorm_bwd_ws(*args, _p(dgamma), _p(dbeta), rows, cols, _p(ws), ws.numel(), _stream())
        _check(rc, "mt_layernorm_bwd_ws", 2)
        if twin is not None:
            dx._mt_bf16 = twin
        return dx, dgamma, dbeta
    if want_wgrad:
        dgb = torch.zeros((2, cols), device=x.device, dtype=torch.float32)   # one fill for both accumulators
        dgamma, dbeta = dgb[0], dgb[1]
    rc = lib.mt_layernorm_bwd(*args, _p(dgamma), _p(dbeta), rows, cols, _stream())
    _check(rc, "mt_layernorm_bwd")
    if twin is not None:
        dx._mt_bf16 = twin
    return dx, dgamma, dbeta


def _as_compute(t: torch.Tensor, cdt: torch.dtype) -> torch.Tensor:
    """``t`` in the compute dtype: the bf16 twin written by the producing LayerNorm backward when there is one (the
    attribute travels with the tensor object through autograd), else a cast pass."""
    if cdt == torch.float32:
        return t
    twin = getattr(t, "_mt_bf16", None)
    if twin is not None and cdt == torch.bfloat16 and twin.shape == t.shape:
        return twin
    return cast(t, cdt)


class DropSpec:
    """Train-mode Dropout(p) + DropPath of one residual branch of the frozen encoder (``mt_dropout``): the keep mask of
    element i comes from a counter RNG keyed by ``seed`` (device int64 [1]) and ``stream_id``; ``path_scale`` is the
    device fp32 [1] DropPath factor (0 or 1 / keep) or None.  Nothing is stored: the backward regenerates the mask."""

    def __init__(self, p: float, seed: torch.Tensor, stream_id: int, path_scale: Optional[torch.Tensor] = None):
        assert 0.0 <= p < 1.0 and seed.dtype == torch.int64 and seed.is_cuda and seed.numel() == 1
        assert path_scale is None or (path_scale.dtype == torch.float32 and path_scale.is_cuda and path_scale.numel() == 1)
        self.p, self.seed, self.stream_id, self.path_scale = float(p), seed, int(stream_id), path_scale
        self.c_struct = _lib.Dropout(self.p, seed.data_ptr(), self.stream_id,
                                     path_scale.data_ptr() if path_scale is not None else None)

    def ref(self):
        return ctypes.byref(self.c_struct)


def _drop(d: Optional[DropSpec]):
    return d.ref() if d is not None else None


def add_layernorm_fwd(x, a, gamma, beta, out_dtype, eps: float = LN_EPS, abias=None, drop: Optional[DropSpec] = None):
    """x_out = x + D(a [+ abias]) (fp32), y = LN(x_out); D = train-mode dropout / DropPath (identity when drop is None)."""
    rows, cols = x.shape
    assert x.dtype == torch.float32
    x_out = torch.empty_like(x)
    y = torch.empty((rows, cols), device=x.device, dtype=out_dtype)
    mean = torch.empty(rows, device=x.device, dtype=torch.float32)
    rstd = torch.empty(rows, device=x.device, dtype=torch.float32)
    rc = _lib.load().mt_add_layernorm_fwd(_p(x), _p(a), _dt(a), _p(abias), _p(gamma), _p(beta), _p(x_out), _p(y), _dt(y),
                                          _p(mean), _p(rstd), rows, cols, eps, _drop(drop), _stream())
    _check(rc, "mt_add_layernorm_fwd")
    return x_out, y, mean, rstd


def gelu_ln_fwd(h, gamma, beta, out_dtype, eps: float = LN_EPS, hbias=None):
    rows, cols = h.shape
    y = torch.empty((rows, cols), device=h.device, dtype=out_dtype)
    mean = torch.empty(rows, device=h.device, dtype=torch.float32)
    rstd = torch.empty(rows, device=h.device, dtype=torch.float32)
    rc = _lib.load().mt_gelu_ln_fwd(_p(h), _dt(h), _p(hbias), _p(gamma), _p(beta), _p(y), _dt(y), _p(mean), _p(rstd), rows,
                                    cols, eps, _stream())
    _check(rc, "mt_gelu_ln_fwd")
    return y, mean, rstd


def gelu_ln_bwd(dy, h, gamma, mean, rstd, out_dtype, hbias=None):
    rows, cols = h.shape
    dh = torch.empty((rows, cols), device=h.device, dtype=out_dtype)
    rc = _lib.load().mt_gelu_ln_bwd(_p(dy), _dt(dy), _p(h), _dt(h), _p(hbias), _p(gamma), _p(mean), _p(rstd), _p(dh),
                                    _dt(dh), rows, cols, _stream())
    _check(rc, "mt_gelu_ln_bwd")
    return dh


def residual_bias_add(x, a, bias, drop: Optional[DropSpec] = None):
    """y = x + D(a + bias) (fp32 residual stream)."""
    rows, cols = x.shape
    y = torch.empty_like(x)
    rc = _lib.load().mt_residual_bias_add(_p(x), _p(a), _dt(a), _p(bias), _p(y), rows, cols, _drop(drop), _stream())
    _check(rc, "mt_residual_bias_add")
    return y


def dropout_bwd_cast(src: torch.Tensor, dtype: torch.dtype, drop: DropSpec) -> torch.Tensor:
    """Gradient of a dropped branch: src * keep_mask / (1 - p) * path_scale in ``dtype`` (same mask as the forward)."""
    dst = torch.empty(src.shape, device=src.device, dtype=dtype)
    rc = _lib.load().mt_dropout_bwd_cast(_p(src), _dt(src), _p(dst), _dt(dst), src.numel(), drop.ref(), _stream())
    _check(rc, "mt_dropout_bwd_cast")
    return dst


def dilated_attn_fwd(geom: Geometry, qkv: torch.Tensor, impl: int):
    """qkv [n_alloc, 3E] -> (o_br [o_elems], lse_br [lse_elems]) in the compact per-branch layout."""
    o_br = torch.empty(geom.o_elems, device=qkv.device, dtype=qkv.dtype)
    lse_br = torch.empty(geom.lse_elems, device=qkv.device, dtype=torch.float32)
    with _timed("dilated_attn_fwd"):
        rc = _lib.load().mt_dilated_attn_fwd(geom.ref(), _p(qkv), qkv.stride(0), qkv.shape[0], _dt(qkv), _p(o_br),
                                             _p(lse_br), impl, _stream())
    _check(rc, "mt_dilated_attn_fwd")
    return o_br, lse_br


def dilated_merge_ln_fwd(geom: Geometry, o_br, lse_br, gamma, beta, eps: float = LN_EPS, want_attn: bool = False):
    N, E = geom.n_tokens, geom.heads * geom.head_dim
    y = torch.empty((N, E), device=o_br.device, dtype=o_br.dtype)
    attn = torch.empty((N, E), device=o_br.device, dtype=o_br.dtype) if want_attn else None
    lse = torch.empty((N, geom.heads), device=o_br.device, dtype=torch.float32)
    mean = torch.empty(N, device=o_br.device, dtype=torch.float32)
    rstd = torch.empty(N, device=o_br.device, dtype=torch.float32)
    rc = _lib.load().mt_dilated_merge_ln_fwd(geom.ref(), _p(o_br), _p(lse_br), _dt(o_br), _p(attn), _p(lse), _p(gamma),
                                             _p(beta), eps, _p(y), _p(mean), _p(rstd), _stream())
    _check(rc, "mt_dilated_merge_ln_fwd")
    return y, attn, lse, mean, rstd


def dilated_merge_ln_bwd(geom: Geometry, dy, o_br, lse_br, gamma, mean, rstd):
    N, E = geom.n_tokens, geom.heads * geom.head_dim
    # n_alloc rows with a zero tail: the tcgen05 backward reads dO tiles through TMA like the qkv buffer
    dattn = torch.empty((geom.n_alloc, E), device=o_br.device, dtype=o_br.dtype)
    if geom.n_alloc > N:
        dattn[N:].zero_()
    delta_br = torch.empty(geom.lse_elems, device=o_br.device, dtype=torch.float32)
    rc = _lib.load().mt_dilated_merge_ln_bwd(geom.ref(), _p(dy), _dt(dy), _p(o_br), _p(lse_br), _p(gamma), _p(mean),
                                             _p(rstd), _dt(o_br), _p(dattn), _p(delta_br), _stream())
    _check(rc, "mt_dilated_merge_ln_bwd")
    return dattn, delta_br


def dilated_bwd_impl(impl: int) -> int:
    """The backward kernel that runs for the requested ``impl``: in deterministic mode the tcgen05 backward (1, 2) runs
    as impl 4, the deterministic one; the SIMT backward (0) has no deterministic variant and raises there."""
    from . import config
    if impl == 0:
        config.check_deterministic("the SIMT dilated-attention backward (fp32 mode, or attn_impl simt)")
    elif impl in (1, 2) and config.deterministic():
        return config.DETERMINISTIC_BWD_IMPL
    return impl


def dilated_attn_bwd(geom: Geometry, qkv, dattn, lse, delta_br, impl: int):
    """dattn [n_alloc, E] (rows >= N zero), merged lse [N, H], per-branch delta -> dqkv fp32 [N, 3E]."""
    N, E = geom.n_tokens, geom.heads * geom.head_dim
    assert dattn.shape[0] == geom.n_alloc, "dattn must have n_alloc rows (zero tail), see dilated_merge_ln_bwd"
    impl = dilated_bwd_impl(impl)
    dqkv = torch.empty((geom.n_alloc, 3 * E), device=qkv.device, dtype=torch.float32)  # rows >= N: reduce scratch
    with _timed("dilated_attn_bwd"):
        rc = _lib.load().mt_dilated_attn_bwd(geom.ref(), _p(qkv), qkv.stride(0), qkv.shape[0], _p(dattn), _p(lse),
                                             _p(delta_br), _dt(qkv), _p(dqkv), impl, _stream())
    # memset + kernel; the deterministic backward (impl 4) launches a dQ and a dK / dV kernel per branch
    _check(rc, "mt_dilated_attn_bwd", 1 + (2 * len(geom.ratios) if impl == 4 else 1))
    return dqkv[:N]


def _rows_ok(t: torch.Tensor) -> None:
    assert t.is_cuda and t.dim() == 2 and t.stride(1) == 1 and t.stride(0) % 8 == 0 and t.data_ptr() % 16 == 0, \
        "cross-attention operands: CUDA [rows, cols] views with unit column stride and 16-byte aligned rows"


def _ptr(t: torch.Tensor):
    return ctypes.c_void_p(t.data_ptr())


def cross_impl(t: torch.Tensor) -> int:
    """``impl`` of mt_cross_attn_*: TF32 tensor cores for fp32 tensors in bf16 mode, exact fp32 SIMT math otherwise."""
    from . import config
    return 1 if (config.mode() == "bf16" and t.dtype == torch.float32 and config.flag("cross_tc")) else 0


def cross_attn_fwd(q, k, v, heads: int, impl: Optional[int] = None):
    """q [Lq, E'], k / v [Lk, E'] (row-strided views allowed: e.g. the halves of one [Lk, 2E'] buffer) -> o, lse."""
    lq, e = q.shape
    lk = k.shape[0]
    hd = e // heads
    for t in (q, k, v):
        _rows_ok(t)
    assert k.stride(0) == v.stride(0) and k.dtype == q.dtype == v.dtype
    impl = cross_impl(q) if impl is None else impl
    o = torch.empty((lq, e), device=q.device, dtype=q.dtype)
    lse = torch.empty((lq, heads), device=q.device, dtype=torch.float32)
    lib = _lib.load()
    nws = lib.mt_cross_attn_workspace_floats(lq, lk, heads, hd, _dt(q), impl)
    ws = torch.empty(max(int(nws), 1), device=q.device, dtype=torch.float32)
    rc = lib.mt_cross_attn_fwd(_ptr(q), q.stride(0), _ptr(k), _ptr(v), k.stride(0), _dt(q), _ptr(o), o.stride(0), _p(lse),
                               lq, lk, heads, hd, _p(ws), int(nws), impl, _stream())
    _check(rc, "mt_cross_attn_fwd", 2 if nws else 1)
    return o, lse


def cross_attn_probs(q, k, lse, heads: int, impl: Optional[int] = None):
    """Head-averaged attention probabilities [Lq, Lk] fp32 of the ``cross_attn_fwd`` call that took ``q``, ``k`` (row-
    strided views allowed) and returned ``lse``: nn.MultiheadAttention's ``need_weights=True`` output.  Pass the same
    ``impl`` as that forward (default: the same selection)."""
    lq, e = q.shape
    lk = k.shape[0]
    for t in (q, k):
        _rows_ok(t)
    assert k.dtype == q.dtype and lse.dtype == torch.float32 and lse.shape == (lq, heads) and lse.is_contiguous()
    impl = cross_impl(q) if impl is None else impl
    p = torch.empty((lq, lk), device=q.device, dtype=torch.float32)
    with _timed("cross_attn_probs"):
        rc = _lib.load().mt_cross_attn_probs(_ptr(q), q.stride(0), _ptr(k), k.stride(0), _dt(q), _p(lse), _p(p),
                                             p.stride(0), lq, lk, heads, e // heads, impl, _stream())
    _check(rc, "mt_cross_attn_probs")
    return p


def cross_attn_bwd(q, k, v, o, d_o, lse, heads: int, impl: Optional[int] = None, packed_kv: bool = False):
    """-> dq [Lq, E'], dk, dv [Lk, E'] fp32.  ``packed_kv``: dk / dv are the two halves of ONE [Lk, 2E'] buffer (returned
    as views), the layout the gradient of a fused k|v projection wants."""
    lq, e = q.shape
    lk = k.shape[0]
    for t in (q, k, v, o, d_o):
        _rows_ok(t)
    assert k.stride(0) == v.stride(0) and o.stride(0) == d_o.stride(0)
    impl = cross_impl(q) if impl is None else impl
    det = _deterministic()
    if det and impl == 0:
        from . import config
        config.check_deterministic("the SIMT cross-attention backward (fp32 mode, or cross_tc off)")
        det = False   # warn_only: the warning is all torch's flag asks for
    dq = torch.empty((lq, e), device=q.device, dtype=torch.float32)
    if packed_kv:
        dkv = torch.empty((lk, 2 * e), device=q.device, dtype=torch.float32)
        dk, dv = dkv[:, :e], dkv[:, e:]
    else:
        dk = torch.empty((lk, e), device=q.device, dtype=torch.float32)
        dv = torch.empty((lk, e), device=q.device, dtype=torch.float32)
    lib = _lib.load()
    args = (_ptr(q), q.stride(0), _ptr(k), _ptr(v), k.stride(0), _ptr(o), _ptr(d_o), o.stride(0), _p(lse), _dt(q), _ptr(dq),
            dq.stride(0), _ptr(dk), _ptr(dv), dk.stride(0), lq, lk, heads, e // heads)
    if det:
        # split loops store partials that a second pass sums in split order (no atomics); workspace from the graph's
        # pool under capture
        nws = int(lib.mt_cross_attn_bwd_workspace_floats(lq, lk, heads, e // heads, _dt(q), impl))
        ws = torch.empty(max(nws, 4), device=q.device, dtype=torch.float32)
        rc = lib.mt_cross_attn_bwd_ws(*args, _p(ws), nws, impl, _stream())
        _check(rc, "mt_cross_attn_bwd_ws", 2 if nws else 1)
        return dq, dk, dv
    rc = lib.mt_cross_attn_bwd(*args, impl, _stream())
    _check(rc, "mt_cross_attn_bwd", 5)
    return dq, dk, dv


def linear_sm100(a: torch.Tensor, w: torch.Tensor, mode: int = _lib.MT_EPI_PLAIN, bias=None, residual=None,
                 want_f32: bool = True, want_bf16: bool = False, stats=None, col_c1=None, col_c2=None, ln_cols: int = 0,
                 eps: float = LN_EPS, out_f32=None, out_bf16=None, ln_mean_out=None, ln_rstd_out=None, impl: int = 0,
                 out_aux=None, in_u=None, in_g=None):
    """C = A W^T on the tcgen05 tensor cores with a fused epilogue (``mt_linear_sm100``): a [M, K] bf16, w [N, K] bf16
    (nn.Linear layout).  Returns (out_f32 or None, out_bf16 or None).  See include/modaltune_b200.h for the modes."""
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and a.dim() == 2 and w.dim() == 2
    assert a.stride(1) == 1 and w.stride(1) == 1 and a.shape[1] == w.shape[1]
    M, K = a.shape
    N = w.shape[0]
    if out_f32 is None and want_f32:
        out_f32 = torch.empty((M, N), device=a.device, dtype=torch.float32)
    if out_bf16 is None and want_bf16:
        out_bf16 = torch.empty((M, N), device=a.device, dtype=torch.bfloat16)
    ep = _lib.LinearEpilogue()
    ep.mode, ep.ln_cols, ep.ln_eps, ep.impl = int(mode), int(ln_cols), float(eps), int(impl)
    ptr = lambda t: t.data_ptr() if t is not None else None
    for t in (bias, residual, col_c1, col_c2, stats):
        assert t is None or (t.is_cuda and t.dtype == torch.float32)
    ep.bias, ep.residual, ep.col_c1, ep.col_c2, ep.stats = ptr(bias), ptr(residual), ptr(col_c1), ptr(col_c2), ptr(stats)
    ep.out_f32, ep.out_bf16 = ptr(out_f32), ptr(out_bf16)
    ep.ln_mean_out, ep.ln_rstd_out = ptr(ln_mean_out), ptr(ln_rstd_out)
    for t in (out_aux, in_u, in_g):
        assert t is None or (t.is_cuda and t.dtype == torch.bfloat16 and t.is_contiguous() and t.shape == (M, N))
    ep.out_aux_bf16, ep.in_u_bf16, ep.in_g_bf16 = ptr(out_aux), ptr(in_u), ptr(in_g)
    ep.ld_out_f32 = out_f32.stride(0) if out_f32 is not None else 0
    ep.ld_out_bf16 = out_bf16.stride(0) if out_bf16 is not None else 0
    ep.ld_residual = residual.stride(0) if residual is not None else 0
    with _timed("linear_sm100"):
        rc = _lib.load().mt_linear_sm100(ctypes.c_void_p(a.data_ptr()), a.stride(0), ctypes.c_void_p(w.data_ptr()),
                                         w.stride(0), M, N, K, ctypes.byref(ep), _stream())
    _check(rc, "mt_linear_sm100")
    return out_f32, out_bf16


def ffn_bwd_prep(dy, y, x1, c1, c2, mean, rstd, ln_cols: int):
    """-> (rowv [rows, 4] = (mean, rstd, m1, m2), dy in bf16): the per-row inputs of the MT_EPI_GELU_LN_BWD epilogue."""
    rows, cols = dy.shape
    for t in (dy, y, x1):
        assert t.dtype == torch.float32 and t.shape == (rows, cols)
    rowv = torch.empty((rows, 4), device=dy.device, dtype=torch.float32)
    dy16 = torch.empty((rows, cols), device=dy.device, dtype=torch.bfloat16)
    rc = _lib.load().mt_ffn_bwd_prep(_p(dy), _p(y), _p(x1), _p(c1), _p(c2), _p(mean), _p(rstd), _p(rowv), _p(dy16), rows,
                                     cols, int(ln_cols), _stream())
    _check(rc, "mt_ffn_bwd_prep")
    return rowv, dy16


def layernorm_bwd_ffn_prep(dy, x, gamma, mean, rstd, residual, below):
    """``layernorm_bwd`` (fp32, 768 columns, residual, bf16 twin) that also forms the FFN-backward row vector of the layer
    BELOW (``mt_layernorm_bwd_ffn_prep``): ``below`` = (x1, c1, c2, mean_f, rstd_f, ln_cols) of that layer.
    -> (dx fp32, dx bf16, rowv [rows, 4])."""
    rows, cols = x.shape
    x1b, c1, c2, mean_f, rstd_f, ln_cols = below
    dx = torch.empty((rows, cols), device=x.device, dtype=torch.float32)
    twin = torch.empty((rows, cols), device=x.device, dtype=torch.bfloat16)
    rowv = torch.empty((rows, 4), device=x.device, dtype=torch.float32)
    rc = _lib.load().mt_layernorm_bwd_ffn_prep(_p(dy), _p(x), _p(gamma), _p(mean), _p(rstd), _p(residual), _p(dx), _p(twin),
                                               _p(x1b), _p(c1), _p(c2), _p(mean_f), _p(rstd_f), _p(rowv), rows, cols,
                                               int(ln_cols), _stream())
    _check(rc, "mt_layernorm_bwd_ffn_prep")
    return dx, twin, rowv


def embed_assemble(proj, bias, coords, table, cls, tile_size: float = 256.0):
    """proj [L, E] (GEMM output), coords [L, 2] -> x [L+1, E] fp32 with the sincos positions and the cls row."""
    L, E = proj.shape
    x = torch.empty((L + 1, E), device=proj.device, dtype=torch.float32)
    rc = _lib.load().mt_embed_assemble(_p(proj), _dt(proj), _p(bias), _p(coords), _p(table), _p(cls), _p(x), L, E,
                                       table.shape[0], float(tile_size), _stream())
    _check(rc, "mt_embed_assemble")
    return x


def colsum(x: torch.Tensor) -> torch.Tensor:
    """x.sum(0) for an fp32 [rows, cols] CUDA tensor (row-strided views allowed): the adapter's bias gradients."""
    rows, cols = x.shape
    if not (x.is_cuda and x.dtype == torch.float32 and x.stride(1) == 1 and cols % 4 == 0 and cols <= 4096
            and x.stride(0) % 4 == 0 and x.data_ptr() % 16 == 0 and rows >= 1024):
        return x.sum(0)            # short inputs (the 66 modal tokens): one library launch instead of memset + kernel
    out = torch.empty(cols, device=x.device, dtype=torch.float32)
    if _deterministic():
        ws = _colreduce_workspace(x.device, cols)
        rc = _lib.load().mt_colsum_ws(ctypes.c_void_p(x.data_ptr()), x.stride(0), _p(out), rows, cols, _p(ws), ws.numel(),
                                      _stream())
        _check(rc, "mt_colsum_ws", 2)
        return out
    rc = _lib.load().mt_colsum(ctypes.c_void_p(x.data_ptr()), x.stride(0), _p(out), rows, cols, _stream())
    _check(rc, "mt_colsum")
    return out


def cast(src: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    dst = torch.empty(src.shape, device=src.device, dtype=dtype)
    rc = _lib.load().mt_cast(_p(src), _dt(src), _p(dst), _dt(dst), src.numel(), _stream())
    _check(rc, "mt_cast")
    return dst


# ---------------------------------------------------------------------------------------------------------------------
# autograd: trainable LayerNorm, cross-attention core, Injector tail
# ---------------------------------------------------------------------------------------------------------------------
class LayerNormFn(torch.autograd.Function):
    """y = LN(x[row0:]) * gamma + beta [+ add]  with x [rows, 768] fp32; y in ``out_dtype``.  Grads for x (full, rows
    < row0 get zero), gamma, beta, add.  ``row0`` lets the adapter normalise the tile tokens of the [cls | tiles] buffer
    in place: no slice / concat copies of the [N, 768] stream, forward or backward."""

    @staticmethod
    def forward(ctx, x, gamma, beta, add, out_dtype, row0):
        x = x.contiguous()
        xv = x[row0:] if row0 else x
        g32, b32 = _f32(gamma).contiguous(), _f32(beta).contiguous()
        addc = None
        if add is not None:
            assert add.shape == xv.shape
            addc = add.contiguous()
        y, mean, rstd = layernorm_fwd(xv, g32, b32, out_dtype, add=addc)
        ctx.save_for_backward(x, g32, mean, rstd)
        ctx.has_add = add is not None
        ctx.add_dtype = add.dtype if add is not None else None
        ctx.need_w = gamma.requires_grad or beta.requires_grad
        ctx.row0 = row0
        return y

    @staticmethod
    def backward(ctx, dy):
        x, g32, mean, rstd = ctx.saved_tensors
        dy = dy.contiguous()
        row0 = ctx.row0
        if row0:
            dx = torch.empty_like(x)
            dx[:row0].zero_()
            _, dgamma, dbeta = layernorm_bwd(dy, x[row0:], g32, mean, rstd, x.dtype, want_wgrad=ctx.need_w,
                                             out=dx[row0:])
        else:
            dx, dgamma, dbeta = layernorm_bwd(dy, x, g32, mean, rstd, x.dtype, want_wgrad=ctx.need_w)
        dadd = dy.to(ctx.add_dtype) if ctx.has_add else None
        return dx, dgamma, dbeta, dadd, None, None


def layer_norm(x, gamma, beta, add=None, out_dtype=None, row0: int = 0):
    return LayerNormFn.apply(x, gamma, beta, add, out_dtype or x.dtype, row0)


class CrossAttnFn(torch.autograd.Function):
    """softmax(q k^T / sqrt(hd)) v over [L, heads*hd] operands; the core of nn.MultiheadAttention in the adapter.
    ``kv`` None: separate k, v.  Otherwise k | v are the two halves of ``kv`` [Lk, 2 E'] (the output of one fused
    projection GEMM), read in place through row strides, and the gradient comes back as one [Lk, 2 E'] tensor: no split /
    concat copies on either side.  Returns (o, lse [Lq, heads]); lse is not differentiable (``cross_attn_probs`` input)."""

    @staticmethod
    def forward(ctx, q, k, v, kv, heads):
        q = q.contiguous()
        if kv is not None:
            if not (kv.stride(1) == 1 and kv.stride(0) % 8 == 0 and kv.data_ptr() % 16 == 0):
                kv = kv.contiguous()      # a column slice of a wider projection buffer is read in place
            e = q.shape[1]
            k, v = kv[:, :e], kv[:, e:]
        else:
            k, v = k.contiguous(), v.contiguous()
        o, lse = cross_attn_fwd(q, k, v, heads)
        ctx.save_for_backward(q, k, v, o, lse)
        ctx.heads, ctx.packed = heads, kv is not None
        ctx.mark_non_differentiable(lse)
        ctx.set_materialize_grads(False)   # no zero-filled gradient for lse in every backward
        return o, lse

    @staticmethod
    def backward(ctx, d_o, _dlse):
        q, k, v, o, lse = ctx.saved_tensors
        dq, dk, dv = cross_attn_bwd(q, k, v, o, d_o.contiguous().to(q.dtype), lse, ctx.heads, packed_kv=ctx.packed)
        if ctx.packed:
            dkv = dk._base if dk._base is not None else torch.cat([dk, dv], 1)
            return dq.to(q.dtype), None, None, dkv.to(k.dtype), None
        return dq.to(q.dtype), dk.to(k.dtype), dv.to(v.dtype), None, None


def cross_attention(q, k, v, heads: int, return_lse: bool = False):
    o, lse = CrossAttnFn.apply(q, k, v, None, heads)
    return (o, lse) if return_lse else o


def cross_attention_kv(q, kv, heads: int, return_lse: bool = False):
    """``cross_attention`` with k | v given as one [Lk, 2 E'] tensor."""
    o, lse = CrossAttnFn.apply(q, None, None, kv, heads)
    return (o, lse) if return_lse else o


def gated_residual_fwd(a, b, g32, out=None):
    y = out if out is not None else torch.empty_like(a)
    rows, cols = a.shape
    rc = _lib.load().mt_gated_residual(_p(a), _p(b), _dt(b), _p(g32), _p(y), rows, cols, _stream())
    _check(rc, "mt_gated_residual")
    return y


def gated_residual_bwd(dy, a, b, g32, out=None, want_dysum: bool = False):
    """-> (da, db, dgate[, dysum = sum_r dy when asked for])"""
    rows, cols = a.shape
    da = out if out is not None else torch.empty_like(a)
    db = torch.empty_like(b)
    dgate = torch.empty(cols, device=a.device, dtype=torch.float32)
    dysum = torch.empty(cols, device=a.device, dtype=torch.float32) if want_dysum else None
    args = (_p(dy), _p(a), _p(b), _dt(b), _p(g32), _p(da), _p(db), _dt(db), _p(dgate), _p(dysum), rows, cols)
    if _deterministic():
        ws = _colreduce_workspace(a.device, cols)
        rc = _lib.load().mt_gated_residual_bwd_ws(*args, _p(ws), ws.numel(), _stream())
        _check(rc, "mt_gated_residual_bwd_ws", 2)
    else:
        rc = _lib.load().mt_gated_residual_bwd(*args, _stream())
        _check(rc, "mt_gated_residual_bwd")
    return (da, db, dgate, dysum) if want_dysum else (da, db, dgate)


class _tf32:
    """Scoped TF32 for the adapter's skinny trainable GEMMs in bf16 mode (10-bit mantissa operands, fp32 storage)."""

    def __enter__(self):
        self.old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True

    def __exit__(self, *exc):
        torch.backends.cuda.matmul.allow_tf32 = self.old
        return False


class LinearTF32Fn(torch.autograd.Function):
    """y = x w^T + b on fp32 tensors with TF32 tensor-core GEMMs in forward AND backward."""

    @staticmethod
    def forward(ctx, x, w, b):
        ctx.save_for_backward(x, w)
        ctx.has_b = b is not None
        with _tf32():
            return torch.nn.functional.linear(x, w, b)

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        with _tf32():
            dx = dy @ w if ctx.needs_input_grad[0] else None
            dw = dy.t() @ x if ctx.needs_input_grad[1] else None
        db = colsum(dy) if ctx.has_b and ctx.needs_input_grad[2] else None
        return dx, dw, db


def linear_tf32(x, w, b):
    return LinearTF32Fn.apply(x, w, b)


class GatedResidualFn(torch.autograd.Function):
    """y[row0:] = a[row0:] + gate * (a[row0:] + b), y[:row0] = a[:row0]: the Injector tail
    ``query + gamma * (query + attn)`` (adapter_modules.py:231,362) applied to the tile rows of the [cls | tiles]
    buffer ``a`` (row0 = 1) or to a plain [L, 768] tensor (row0 = 0)."""

    @staticmethod
    def forward(ctx, a, b, gate, row0):
        a, b = a.contiguous(), b.contiguous()
        g32 = _f32(gate).contiguous()
        if row0:
            y = torch.empty_like(a)
            y[:row0].copy_(a[:row0])
            gated_residual_fwd(a[row0:], b, g32, out=y[row0:])
        else:
            y = gated_residual_fwd(a, b, g32)
        ctx.save_for_backward(a, b, g32)
        ctx.row0 = row0
        return y

    @staticmethod
    def backward(ctx, dy):
        a, b, g32 = ctx.saved_tensors
        dy = dy.contiguous()
        row0 = ctx.row0
        if row0:
            da = torch.empty_like(a)
            da[:row0].copy_(dy[:row0])
            _, db, dgate = gated_residual_bwd(dy[row0:], a[row0:], b, g32, out=da[row0:])
        else:
            da, db, dgate = gated_residual_bwd(dy, a, b, g32)
        return da, db, dgate, None


def gated_residual(a, b, gate, row0: int = 0):
    return GatedResidualFn.apply(a, b, gate, row0)


class SharedKVProjectFn(torch.autograd.Function):
    """k | v projections of SEVERAL Extractors that read the same slide tokens (the last interaction block runs three
    on one ``xfull``, adapter_modules.py:508-516): LayerNorm statistics do not depend on the affine parameters, so with
    ``xhat = normalise(x)`` every extractor's ``LN_e(x) Wkv_e^T + b_e`` is ``xhat (Wkv_e diag gamma_e)^T + (Wkv_e beta_e +
    b_e)``: ONE normalisation pass and ONE GEMM against the stacked, composed weights (formed by the caller with
    differentiable weight-sized ops) instead of three LayerNorms and three GEMMs over [L, 768]; in the backward one
    dX GEMM, one dW GEMM, one affine-free LayerNorm backward, and the slide-token gradient is written once instead of
    being summed from three [N, 768] tensors by autograd.

    x [N, 768] fp32 (rows < row0 are skipped), w [n * 384, 768], b [n * 384]  ->  kv [N - row0, n * 384]."""

    @staticmethod
    def forward(ctx, x, w, b, row0):
        x = x.contiguous()
        xv = x[row0:]
        ones, zeros = _unit_affine(x.device, x.shape[1])
        xhat, mean, rstd = layernorm_fwd(xv, ones, zeros, torch.float32)
        kv = _adapter_addmm(b, xhat, w.t())
        ctx.save_for_backward(x, xhat, w, mean, rstd)
        ctx.row0 = row0
        return kv

    @staticmethod
    def backward(ctx, dkv):
        x, xhat, w, mean, rstd = ctx.saved_tensors
        row0 = ctx.row0
        dkv = dkv.contiguous()
        db = colsum(dkv)
        dw = _adapter_mm(dkv.t(), xhat)
        dxhat = _adapter_mm(dkv, w)
        ones, _ = _unit_affine(x.device, x.shape[1])
        dx = torch.empty_like(x)
        if row0:
            dx[:row0].zero_()
        layernorm_bwd(dxhat, x[row0:], ones, mean, rstd, torch.float32, out=dx[row0:])
        return dx, dw, db, None


_unit_affine_cache: Dict[tuple, tuple] = {}


def _unit_affine(device, cols: int):
    key = (str(device), cols)
    if key not in _unit_affine_cache:
        _unit_affine_cache[key] = (torch.ones(cols, device=device), torch.zeros(cols, device=device))
    return _unit_affine_cache[key]


def shared_kv_project(x, w, b, row0: int = 0):
    return SharedKVProjectFn.apply(x, w, b, row0)


def _adapter_mm(a, b):
    """a @ b for the adapter's skinny GEMMs: TF32 tensor cores in bf16 mode, exact fp32 in fp32 mode."""
    from . import config
    if config.mode() == "bf16" and a.is_cuda:
        with _tf32():
            return a @ b
    return a @ b


def _adapter_addmm(bias, a, bt):
    from . import config
    if config.mode() == "bf16" and a.is_cuda:
        with _tf32():
            return torch.addmm(bias, a, bt)
    return torch.addmm(bias, a, bt)


class InjectorFn(torch.autograd.Function):
    """The whole Injector on the [cls | tiles] buffer as ONE autograd node (adapter_modules.py:338-369 with the
    CrossAttentionLayer of :130-245 inlined):

        y[row0:] = x + gate * (x + attn(LN(x), k, v) Wo^T + bo),   y[:row0] = x[:row0],   x = xfull[row0:]

    ``wq`` [192, 768] / ``bq`` and ``wo`` [768, 192] / ``bo`` are the COMPOSED projections (cffn q_proj then the MHA
    in-projection; MHA out_proj then cffn output_proj: two linear maps with nothing between them), formed by the caller
    with differentiable [192 x 192 x 768] products, so the two [L, 192] intermediates, four of the six backward GEMMs over
    L rows and their bias reductions never exist.  ``kv`` [M, 384] = k | v of the modal tokens.  The backward writes the
    gradient of the residual stream once: the gated tail's ``dy (1 + gate)`` goes into the buffer the LayerNorm backward
    then adds its part to in place (no [N, 768] autograd add, no zero fill), and the bias gradient of the output
    projection comes from the column sums the gated-residual kernel already forms."""

    @staticmethod
    def forward(ctx, x, kv, ln_w, ln_b, wq, bq, wo, bo, gate, row0, heads):
        x = x.contiguous()
        xv = x[row0:]
        kv = kv.contiguous()
        e = wq.shape[0]
        g32, w32, b32 = _f32(gate).contiguous(), _f32(ln_w).contiguous(), _f32(ln_b).contiguous()
        t2, mean, rstd = layernorm_fwd(xv, w32, b32, torch.float32)
        q = _adapter_addmm(bq, t2, wq.t())
        o, lse = cross_attn_fwd(q, kv[:, :e], kv[:, e:], heads)
        a = _adapter_addmm(bo, o, wo.t())
        y = torch.empty_like(x)
        if row0:
            y[:row0].copy_(x[:row0])
        gated_residual_fwd(xv, a, g32, out=y[row0:])
        ctx.save_for_backward(x, kv, w32, wq, wo, g32, mean, rstd, t2, q, o, lse, a)
        ctx.row0, ctx.heads = row0, heads
        return y

    @staticmethod
    def backward(ctx, dy):
        x, kv, w32, wq, wo, g32, mean, rstd, t2, q, o, lse, a = ctx.saved_tensors
        row0, e = ctx.row0, wq.shape[0]
        dy = dy.contiguous()
        xv = x[row0:]
        dx = torch.empty_like(x)
        if row0:
            dx[:row0].copy_(dy[:row0])
        _, db, dgate, dysum = gated_residual_bwd(dy[row0:], xv, a, g32, out=dx[row0:], want_dysum=True)
        dbo = g32 * dysum
        dwo = _adapter_mm(db.t(), o)                       # [768, 192]
        d_o = _adapter_mm(db, wo)                          # [L, 192]
        del db
        dq, dk, dv = cross_attn_bwd(q, kv[:, :e], kv[:, e:], o, d_o, lse, ctx.heads, packed_kv=True)
        dkv = dk._base if dk._base is not None else torch.cat([dk, dv], 1)
        dbq = colsum(dq)
        dwq = _adapter_mm(dq.t(), t2)                      # [192, 768]
        dt2 = _adapter_mm(dq, wq)                          # [L, 768]
        # dx[row0:] = dy (1 + gate) (written above) + LN'(dt2): residual and output are the same buffer
        _, dlnw, dlnb = layernorm_bwd(dt2, xv, w32, mean, rstd, torch.float32, residual=dx[row0:], want_wgrad=True,
                                      out=dx[row0:])
        return dx, dkv, dlnw, dlnb, dwq, dbq, dwo, dbo, dgate, None, None


def injector(x, kv, ln_w, ln_b, wq, bq, wo, bo, gate, row0: int, heads: int):
    return InjectorFn.apply(x, kv, ln_w, ln_b, wq, bq, wo, bo, gate, row0, heads)


# ---------------------------------------------------------------------------------------------------------------------
# the frozen LongNet encoder layer: one autograd node, dX-only backward
# ---------------------------------------------------------------------------------------------------------------------
class FrozenLayerWeights:
    """Derived, read-only copies of one encoder layer's parameters in the layout the kernels want: fused QKV weight
    [2304, 768], GEMM operands in the compute dtype, LayerNorm scales in fp32.  Rebuilt when a source parameter
    changes (``load_state_dict`` / in-place edits bump ``_version``) or moves."""

    def __init__(self):
        self.key = None

    def refresh(self, layer, dtype: torch.dtype):
        sa, ffn = layer.self_attn, layer.ffn
        params = [sa.q_proj.weight, sa.k_proj.weight, sa.v_proj.weight, sa.q_proj.bias, sa.k_proj.bias,
                  sa.v_proj.bias, sa.out_proj.weight, sa.out_proj.bias, sa.inner_attn_ln.weight,
                  sa.inner_attn_ln.bias, layer.self_attn_layer_norm.weight, layer.self_attn_layer_norm.bias,
                  layer.final_layer_norm.weight, layer.final_layer_norm.bias, ffn.fc1.weight, ffn.fc1.bias,
                  ffn.fc2.weight, ffn.fc2.bias, ffn.ffn_layernorm.weight, ffn.ffn_layernorm.bias]
        key = (dtype, tuple((p.data_ptr(), p._version) for p in params))
        if key == self.key:
            return self
        with torch.no_grad():
            d = lambda p: p.detach().to(dtype).contiguous()
            f = lambda p: p.detach().float().contiguous()
            self.w_qkv = torch.cat([d(sa.q_proj.weight), d(sa.k_proj.weight), d(sa.v_proj.weight)], 0).contiguous()
            self.b_qkv = torch.cat([d(sa.q_proj.bias), d(sa.k_proj.bias), d(sa.v_proj.bias)], 0).contiguous()
            self.w_o, self.b_o = d(sa.out_proj.weight), f(sa.out_proj.bias)
            self.w_1, self.b_1 = d(ffn.fc1.weight), f(ffn.fc1.bias)
            self.w_2, self.b_2 = d(ffn.fc2.weight), f(ffn.fc2.bias)
            self.ln1 = (f(layer.self_attn_layer_norm.weight), f(layer.self_attn_layer_norm.bias))
            self.ln2 = (f(layer.final_layer_norm.weight), f(layer.final_layer_norm.bias))
            self.ln_in = (f(sa.inner_attn_ln.weight), f(sa.inner_attn_ln.bias))
            self.ln_ffn = (f(ffn.ffn_layernorm.weight), f(ffn.ffn_layernorm.bias))
            if dtype == torch.bfloat16:
                # ffn_layernorm folded into fc2 (mt_linear_sm100, MT_EPI_LN_RESIDUAL): W2' = W2 diag(gamma), c1 = W2' 1
                # (over the ROUNDED W2', what the tensor cores multiply), c2 = W2 beta + b2 in fp32
                w2 = ffn.fc2.weight.detach().float()
                self.w_2g = (w2 * self.ln_ffn[0][None, :]).to(dtype).contiguous()
                self.c1_2 = self.w_2g.float().sum(1).contiguous()
                self.c2_2 = (w2 @ self.ln_ffn[1] + self.b_2).contiguous()
                self.b_qkv32 = self.b_qkv.float().contiguous()
                # [in, out] copies: the B operand of the dX GEMMs (C = dY W  ==  dY (W^T)^T)
                self.w_qkv_t = self.w_qkv.t().contiguous()
                self.w_o_t = self.w_o.t().contiguous()
                self.w_1_t = self.w_1.t().contiguous()
                self.w_2_t = self.w_2.t().contiguous()
                self.w_2g_t = self.w_2g.t().contiguous()       # [3072, 768]: dX of fc2 with the LayerNorm scale folded in
        self.key = key
        return self


def _linear(x, w, b):
    return torch.nn.functional.linear(x, w, b)


def _linear_f32out(x, w):
    """x @ w^T with 16-bit operands and an fp32 result (cuBLASLt bf16 x bf16 -> f32): every GEMM whose consumer is an
    element-wise kernel keeps its fp32 accumulator instead of rounding the output to bf16.  No bias: cuBLAS has no
    fused bias epilogue for this combination (it costs a broadcast copy + a beta pass), so the bias is added by the
    consuming kernel."""
    if x.dtype == torch.float32:
        return torch.nn.functional.linear(x, w)
    return torch.mm(x, w.t(), out_dtype=torch.float32)


def _matmul_f32out(a, b):
    if a.dtype == torch.float32:
        return torch.matmul(a, b)
    return torch.mm(a, b, out_dtype=torch.float32)


def _qkv_project(h1: torch.Tensor, W: FrozenLayerWeights, geom: Geometry) -> torch.Tensor:
    """QKV GEMM into a buffer with ``n_alloc`` rows whose tail rows are zero (the TMA gather reads them as the
    reference's zero padding, dilated_attention.py:82-111)."""
    N = geom.n_tokens
    qkv = torch.empty((geom.n_alloc, 3 * EMBED), device=h1.device, dtype=h1.dtype)
    torch.addmm(W.b_qkv, h1, W.w_qkv.t(), out=qkv[:N])
    if geom.n_alloc > N:
        qkv[N:].zero_()
    return qkv


def _use_sm100_gemm(cdt: torch.dtype, rng) -> bool:
    """The fused-epilogue tensor-core GEMMs serve bf16 mode in eval (the train-mode dropout sits between a projection
    and its residual add, where the fused epilogue has no mask: train mode keeps the library GEMM + element-wise path)."""
    from . import config
    return cdt == torch.bfloat16 and not rng and config.gemm_impl() == "sm100"


# hand-over between consecutive frozen layers of one task pass (one slot per CUDA stream: the passes run on their own
# streams and their autograd nodes interleave).  A slot is consumed by the NEXT layer call on that stream whether it
# matches or not, and a match needs the very tensor object (held weakly) or a view of it, with an unchanged version
# counter: a stale entry can never meet an unrelated tensor that happens to reuse the address later.
_ffn_fwd_link: Dict[int, tuple] = {}
_ffn_bwd_link: Dict[int, tuple] = {}


def _link_key(t: torch.Tensor) -> int:
    return torch.cuda.current_stream().cuda_stream if t.is_cuda else 0


def _is_view_of(t: torch.Tensor, ref) -> bool:
    """Is ``t`` the tensor ``ref()`` (a weak reference) or a full view of it?  Identity of the OBJECT, not of the address:
    a tensor of a later step that happens to reuse the memory of a dead one never matches."""
    src = ref()
    if src is None:
        return False
    return (t is src or t._base is src) and t.data_ptr() == src.data_ptr() and t.numel() == src.numel()


def _encoder_layer_forward_sm100(x: torch.Tensor, W: FrozenLayerWeights, geom: Geometry, impl):
    """EncoderLayer.forward with every frozen projection on ``mt_linear_sm100`` and its epilogues: bias + bf16 q/k/v into
    the TMA-ready buffer; out_proj + bias + residual -> x1; fc1 + bias + GELU + LayerNorm(3072) statistics; fc2 with the
    LayerNorm folded in + bias + residual -> y.  The [N, 3072] normalised tensor, the fp32 attention / FFN branch outputs
    and the GELU+LN and residual kernels of the library path do not exist here."""
    N = geom.n_tokens
    cdt = torch.bfloat16
    # is x the output of the encoder layer that ran right before on this stream?  Then this layer's backward can prepare
    # that layer's FFN backward in its last kernel (see _encoder_layer_backward_sm100)
    key = _link_key(x)
    link = _ffn_fwd_link.pop(key, None)
    below = link[1] if (link is not None and _is_view_of(x, link[0]) and tuple(x.shape) == tuple(link[0]().shape)) else None
    h1, mean1, rstd1 = layernorm_fwd(x, W.ln1[0], W.ln1[1], cdt)
    qkv = torch.empty((geom.n_alloc, 3 * EMBED), device=x.device, dtype=cdt)
    if geom.n_alloc > N:
        qkv[N:].zero_()
    linear_sm100(h1, W.w_qkv, bias=W.b_qkv32, want_f32=False, out_bf16=qkv[:N])
    del h1
    o_br, lse_br = dilated_attn_fwd(geom, qkv, impl[0])
    a_ln, _, lse, mean_a, rstd_a = dilated_merge_ln_fwd(geom, o_br, lse_br, W.ln_in[0], W.ln_in[1])
    x1, _ = linear_sm100(a_ln, W.w_o, bias=W.b_o, residual=x)                     # x1 = x + out_proj(a_ln)
    del a_ln
    h2, mean2, rstd2 = layernorm_fwd(x1, W.ln2[0], W.ln2[1], cdt)
    stats = torch.empty((N, W.w_1.shape[0] // 128, 2), device=x.device, dtype=torch.float32)   # slab partials
    from . import config
    fused_bwd = config.ffn_bwd_fused()
    if fused_bwd:
        # the backward runs inside fc2's dX GEMM (MT_EPI_GELU_LN_BWD): it wants gelu(h) and gelu'(h) in bf16 (the same
        # bytes as the fp32 h, no erf / exp per element in the backward, and the forward writes 61 MB less)
        f1 = torch.empty((N, W.w_1.shape[0]), device=x.device, dtype=cdt)          # gelu'(h)
        u = torch.empty((N, W.w_1.shape[0]), device=x.device, dtype=cdt)
        linear_sm100(h2, W.w_1, mode=_lib.MT_EPI_GELU_STATS, bias=W.b_1, want_f32=False, out_bf16=u, out_aux=f1, stats=stats)
    else:
        f1, u = linear_sm100(h2, W.w_1, mode=_lib.MT_EPI_GELU_STATS, bias=W.b_1, want_f32=True, want_bf16=True, stats=stats)
    del h2
    mean_f = torch.empty(N, device=x.device, dtype=torch.float32)
    rstd_f = torch.empty(N, device=x.device, dtype=torch.float32)
    y, _ = linear_sm100(u, W.w_2g, mode=_lib.MT_EPI_LN_RESIDUAL, residual=x1, stats=stats, col_c1=W.c1_2, col_c2=W.c2_2,
                        ln_cols=W.w_2g.shape[1], ln_mean_out=mean_f, ln_rstd_out=rstd_f)
    # saved for the backward: f1 = fc1's fp32 output incl. bias (separate GELU'-LN' kernel) or gelu'(h) in bf16 with
    # u = gelu(h) (fused epilogue); y rides along (it is the next layer's saved input anyway: no extra memory)
    saved = (x, mean1, rstd1, qkv, o_br, lse_br, lse, mean_a, rstd_a, x1, mean2, rstd2, f1, mean_f, rstd_f, y,
             u if fused_bwd else None) + (tuple(below[:5]) if below is not None else (None,) * 5)
    if fused_bwd:
        _ffn_fwd_link[key] = (weakref.ref(y), (x1, W.c1_2, W.c2_2, mean_f, rstd_f, W.w_2g.shape[1]))
    return y, saved


def _encoder_layer_backward_sm100(dy: torch.Tensor, saved, W: FrozenLayerWeights, geom: Geometry, impl):
    (x, mean1, rstd1, qkv, o_br, lse_br, lse, mean_a, rstd_a, x1, mean2, rstd2, f1, mean_f, rstd_f, y, u) = saved[:17]
    below = saved[17:22]
    cdt = torch.bfloat16
    dy = dy.contiguous()
    key = _link_key(dy)
    hand = _ffn_bwd_link.pop(key, None)
    if u is not None:
        # GELU' . LayerNorm' inside the epilogue of fc2's dX GEMM: the two row means of the LayerNorm backward are dot
        # products of [N, 768] tensors, so the fp32 [N, 3072] gradient is never written or read.  When dy was produced by
        # the backward of the layer above on this stream, that layer's last kernel has formed them already (hand-over by
        # storage identity: autograd passes the gradient on through view nodes, which keep pointer and version)
        if (hand is not None and _is_view_of(dy, hand[0]) and hand[1] == dy._version
                and tuple(dy.shape) == tuple(hand[0]().shape)):
            rowv, d_f2 = hand[2], hand[3]
        else:
            rowv, d_f2 = ffn_bwd_prep(dy, y, x1, W.c1_2, W.c2_2, mean_f, rstd_f, W.w_2g.shape[1])
        _, d_f1 = linear_sm100(d_f2, W.w_2g_t, mode=_lib.MT_EPI_GELU_LN_BWD, in_u=u, in_g=f1, stats=rowv, want_f32=False,
                               want_bf16=True)
    else:
        d_f2 = _as_compute(dy, cdt)
        dg, _ = linear_sm100(d_f2, W.w_2_t)                                       # fp32 [N, 3072]
        d_f1 = gelu_ln_bwd(dg, f1, W.ln_ffn[0], mean_f, rstd_f, cdt, hbias=None)
        del dg
    dh2, _ = linear_sm100(d_f1, W.w_1_t)                                          # fp32 [N, 768]
    del d_f1
    dx1, _, _ = layernorm_bwd(dh2, x1, W.ln2[0], mean2, rstd2, torch.float32, residual=dy, bf16_twin=True)
    del dh2
    d_aln, _ = linear_sm100(_as_compute(dx1, cdt), W.w_o_t)                       # fp32 [N, 768]
    dattn, delta_br = dilated_merge_ln_bwd(geom, d_aln, o_br, lse_br, W.ln_in[0], mean_a, rstd_a)
    del d_aln
    dqkv = dilated_attn_bwd(geom, qkv, dattn, lse, delta_br, impl[1])             # fp32 [N, 2304]
    dh1, _ = linear_sm100(cast(dqkv, cdt), W.w_qkv_t)
    if below[0] is not None:
        # x is the output of the layer below: form ITS FFN-backward row vector and bf16 gradient here (one more read)
        dx, twin, rowv_b = layernorm_bwd_ffn_prep(dh1, x, W.ln1[0], mean1, rstd1, dx1, tuple(below) + (W.w_2g.shape[1],))
        _ffn_bwd_link[key] = (weakref.ref(dx), dx._version, rowv_b, twin)
    else:
        dx, _, _ = layernorm_bwd(dh1, x, W.ln1[0], mean1, rstd1, torch.float32, residual=dx1)
    return dx


def encoder_layer_forward(x: torch.Tensor, W: FrozenLayerWeights, geom: Geometry, cdt: torch.dtype, impl, rng=None):
    """x [N, 768] fp32 -> (y fp32, saved tensors); ``impl`` = (forward, backward) attention kernel selectors.
    EncoderLayer.forward (encoder.py:121-175); ``rng`` = (DropSpec of the attention branch, DropSpec of the FFN branch)
    in train mode, None in eval mode."""
    if _use_sm100_gemm(cdt, rng):
        return _encoder_layer_forward_sm100(x, W, geom, impl)
    h1, mean1, rstd1 = layernorm_fwd(x, W.ln1[0], W.ln1[1], cdt)
    qkv = _qkv_project(h1, W, geom)
    del h1
    o_br, lse_br = dilated_attn_fwd(geom, qkv, impl[0])
    a_ln, _, lse, mean_a, rstd_a = dilated_merge_ln_fwd(geom, o_br, lse_br, W.ln_in[0], W.ln_in[1])
    attn_out = _linear_f32out(a_ln, W.w_o)                   # fp32 [N, 768], bias added by the consumer
    del a_ln
    x1, h2, mean2, rstd2 = add_layernorm_fwd(x, attn_out, W.ln2[0], W.ln2[1], cdt, abias=W.b_o,
                                             drop=rng[0] if rng else None)
    del attn_out
    f1 = _linear_f32out(h2, W.w_1)                           # fp32 [N, 3072] WITHOUT fc1's bias, kept for the backward
    del h2
    g, mean_f, rstd_f = gelu_ln_fwd(f1, W.ln_ffn[0], W.ln_ffn[1], cdt, hbias=W.b_1)
    f2 = _linear_f32out(g, W.w_2)
    del g
    y = residual_bias_add(x1, f2, W.b_2, drop=rng[1] if rng else None)
    saved = (x, mean1, rstd1, qkv, o_br, lse_br, lse, mean_a, rstd_a, x1, mean2, rstd2, f1, mean_f, rstd_f)
    return y, saved


def encoder_layer_backward(dy: torch.Tensor, saved, W: FrozenLayerWeights, geom: Geometry, cdt: torch.dtype, impl,
                           rng=None):
    """dX of the frozen layer (no weight gradients: every parameter of the slide encoder is frozen,
    longvit_adapter.py:78-80).  ``rng``: the DropSpecs of the forward (the masks are regenerated, not stored)."""
    if _use_sm100_gemm(cdt, rng):
        return _encoder_layer_backward_sm100(dy, saved, W, geom, impl)
    (x, mean1, rstd1, qkv, o_br, lse_br, lse, mean_a, rstd_a, x1, mean2, rstd2, f1, mean_f, rstd_f) = saved
    dy = dy.contiguous()
    if rng:
        d_f2 = dropout_bwd_cast(dy, cdt, rng[1])
    else:
        d_f2 = _as_compute(dy, cdt)
    dg = _matmul_f32out(d_f2, W.w_2)                                 # fp32 [N, 3072]
    d_f1 = gelu_ln_bwd(dg, f1, W.ln_ffn[0], mean_f, rstd_f, cdt, hbias=W.b_1)
    del dg
    dh2 = _matmul_f32out(d_f1, W.w_1)                                # fp32 [N, 768]
    del d_f1
    twin = cdt == torch.bfloat16 and not rng
    dx1, _, _ = layernorm_bwd(dh2, x1, W.ln2[0], mean2, rstd2, torch.float32, residual=dy, bf16_twin=twin)
    del dh2
    if rng:
        d_out = dropout_bwd_cast(dx1, cdt, rng[0])
    else:
        d_out = _as_compute(dx1, cdt)
    d_aln = _matmul_f32out(d_out, W.w_o)                             # fp32 [N, 768]
    dattn, delta_br = dilated_merge_ln_bwd(geom, d_aln, o_br, lse_br, W.ln_in[0], mean_a, rstd_a)
    del d_aln
    dqkv = dilated_attn_bwd(geom, qkv, dattn, lse, delta_br, impl[1])   # fp32 [N, 2304]
    dqkv_c = dqkv if cdt == torch.float32 else cast(dqkv, cdt)
    dh1 = _matmul_f32out(dqkv_c, W.w_qkv)
    dx, _, _ = layernorm_bwd(dh1, x, W.ln1[0], mean1, rstd1, torch.float32, residual=dx1)
    return dx


class FrozenEncoderLayerFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, W, geom, cdt, impl, rng):
        y, saved = encoder_layer_forward(x.contiguous(), W, geom, cdt, impl, rng)
        ctx.save_for_backward(*saved)
        ctx.W, ctx.geom, ctx.cdt, ctx.impl, ctx.rng = W, geom, cdt, impl, rng
        return y

    @staticmethod
    def backward(ctx, dy):
        dx = encoder_layer_backward(dy, ctx.saved_tensors, ctx.W, ctx.geom, ctx.cdt, ctx.impl, ctx.rng)
        return dx, None, None, None, None, None


def frozen_encoder_layer(x, W, geom, cdt, impl, rng=None):
    if torch.is_grad_enabled() and x.requires_grad:
        return FrozenEncoderLayerFn.apply(x, W, geom, cdt, impl, rng)
    y, _ = encoder_layer_forward(x.contiguous(), W, geom, cdt, impl, rng)
    return y


def train_rng(device, dropout: float, drop_path: float, stream_base: int):
    """The two DropSpecs of one encoder-layer call in train mode: a fresh 64-bit seed and the DropPath factors of the
    attention and FFN branches drawn on the device with torch's generator (graph-capture safe: a captured step redraws
    them on every replay).  timm's drop_path (per sample, scaled by 1 / keep) with batch 1 is one Bernoulli per branch."""
    seed = torch.randint(0, 2 ** 62, (1,), device=device, dtype=torch.int64)
    if drop_path > 0.0:
        keep = 1.0 - drop_path
        scales = (torch.rand(2, device=device) < keep).float() / keep
        ps = (scales[0:1], scales[1:2])
    else:
        ps = (None, None)
    return DropSpec(dropout, seed, stream_base, ps[0]), DropSpec(dropout, seed, stream_base + 1, ps[1])


def attention_flops(geom: Geometry) -> Tuple[float, float]:
    """(forward, backward) algorithmic attention FLOPs of one layer (SURVEY.md §8d)."""
    return geom.flops_fwd, 2.5 * geom.flops_fwd
