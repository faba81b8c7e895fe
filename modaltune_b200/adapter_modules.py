"""Modal Adapter blocks (Multi-Modal Feature Injector / Extractor) on the modaltune_b200 kernels.

Same classes, constructor signatures, ``forward`` signatures and parameter names as the reference's
``models/vitadapter/adapter_modules.py`` (SelfAttentionLayer :18-99, CrossAttentionLayer :130-245, FFNLayer :248-293,
Extractor :296-335, Injector :338-369, InteractionBlockWithCls :372-456, InteractionBlockWithCls_LongNetViT :459-523),
so reference checkpoints load and ``LongNetGene*Adapter.forward`` drives them unchanged.

What runs where: LayerNorm (+ fused positional add), the 12-head x 16 softmax(QK^T/4)V core (smem-resident K/V for the
Injector's many-queries/few-keys shape, split-K + LSE combine for the Extractor's few-queries/many-keys shape) and the
gated residual tail are hand-written kernels (``ops.LayerNormFn`` / ``CrossAttnFn`` / ``GatedResidualFn``); the skinny
trainable projections (768<->192) are cuBLAS GEMMs through autograd.  The reference's ``nn.MultiheadAttention`` call
materialises [12, Lq, Lk] probabilities and their head average (discarded, :225-229); nothing of that size exists here,
except the [Lq, Lk] head average when a forward hook on the attention module asks for it (``MultiheadAttention``).
"""
from __future__ import annotations

import contextlib
from typing import List, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import config, ops


class DropPath(nn.Module):
    """models/vitadapter/drop_path.py:16-37 -- per-sample stochastic depth."""

    def __init__(self, drop_prob: float = 0.0):
        super().__init__()
        self.drop_prob = drop_prob

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1 - self.drop_prob
        mask = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
        if keep > 0.0:
            mask.div_(keep)
        return x * mask


class Identity_mod(nn.Module):
    def __init__(self, *args, **kwargs) -> None:
        super().__init__()

    def forward(self, input, *args, **kwargs):
        return input


def _lin(x, w, b):
    """The adapter's skinny trainable projections (768 <-> 192) on fp32 activations: exact fp32 GEMMs in fp32 mode,
    TF32 tensor-core GEMMs (forward and backward) in bf16 mode.  They are ~0.6% of the step's FLOPs; keeping them and
    the adapter's activations out of bf16 is what keeps the per-parameter gradient cosine above 0.999 (DESIGN.md)."""
    if config.mode() == "bf16" and x.is_cuda:
        return ops.linear_tf32(x, w, b)
    return F.linear(x, w, b)


def _mha_core(mha: nn.MultiheadAttention, query, key, value, need_weights: bool = False):
    """The arithmetic of ``nn.MultiheadAttention(E', heads, kdim=vdim=768, batch_first)`` with separate q/k/v weights
    on 2-D operands: in-projections, softmax(QK^T/sqrt(hd))V (kernel), out-projection.  ``need_weights``: also return the
    head-averaged probabilities [Lq, Lk] fp32 (detached), recomputed by ``ops.cross_attn_probs`` from the forward's q, k
    and lse."""
    e = mha.embed_dim
    b = mha.in_proj_bias
    q = _lin(query, mha.q_proj_weight, b[:e])
    if key is value:
        kv = _lin(key, torch.cat([mha.k_proj_weight, mha.v_proj_weight], 0), b[e:])
        # k | v read in place, gradient returned as one tensor
        o, lse = ops.cross_attention_kv(q, kv, mha.num_heads, return_lse=True)
        k = kv[:, :e]
    else:
        k = _lin(key, mha.k_proj_weight, b[e:2 * e])
        v = _lin(value, mha.v_proj_weight, b[2 * e:])
        o, lse = ops.cross_attention(q, k, v, mha.num_heads, return_lse=True)
    out = _lin(o, mha.out_proj.weight, mha.out_proj.bias)
    if not need_weights:
        return out
    with torch.no_grad():
        return out, ops.cross_attn_probs(q.detach(), k.detach(), lse, mha.num_heads)


# tensors returned to forward hooks while a task pass runs on a side stream (``recording_outputs``)
_side_outputs: Optional[List[torch.Tensor]] = None


@contextlib.contextmanager
def recording_outputs(sink: List[torch.Tensor]):
    """Inside the block, every tensor a ``MultiheadAttention`` forward returns is appended to ``sink``: the caller that
    ran the block on a side stream makes them safe to use on its own stream (``record_stream``)."""
    global _side_outputs
    old, _side_outputs = _side_outputs, sink
    try:
        yield
    finally:
        _side_outputs = old


class MultiheadAttention(nn.MultiheadAttention):
    """``nn.MultiheadAttention`` (same parameters, names and state dict) whose ``forward`` runs the adapter's kernels.

    The adapter layers call ``_mha_core`` directly; they go through this module (``nn.Module.__call__``, so torch's hook
    semantics apply, including a hook that replaces the output) only when it has forward hooks or forward pre-hooks.
    The hooks then receive what the reference's ``need_weights=True`` call returns: ``(attn_output [1, Lq, E'],
    attn_weights [1, Lq, Lk])``, the weights averaged over the heads, fp32 and detached (no autograd history).  Global
    hooks (``nn.modules.module.register_module_forward_hook``) do not reroute the layers."""

    def forward(self, query, key, value, key_padding_mask=None, need_weights=True, attn_mask=None,
                average_attn_weights=True, is_causal=False):
        if key_padding_mask is not None or attn_mask is not None or is_causal:
            raise NotImplementedError("modaltune_b200 MultiheadAttention: key_padding_mask, attn_mask and is_causal are "
                                      "not supported (the ModalTune adapter never uses them)")
        if need_weights and not average_attn_weights:
            raise NotImplementedError("modaltune_b200 MultiheadAttention: per-head weights (average_attn_weights=False) "
                                      "are not supported; only the head average is computed")
        assert self.batch_first, "modaltune_b200 MultiheadAttention takes batch-first [1, L, E] inputs"
        k = _rows(key)
        res = _mha_core(self, _rows(query), k, k if value is key else _rows(value), need_weights)
        out, w = (res[0].unsqueeze(0), res[1].unsqueeze(0)) if need_weights else (res.unsqueeze(0), None)
        if _side_outputs is not None:
            _side_outputs.extend(t for t in (out, w) if t is not None)
        return out, w


def _hooked(m: nn.Module) -> bool:
    return bool(m._forward_hooks or m._forward_pre_hooks)


def hooked_attention(modules) -> List[str]:
    """Names of the adapter attention modules among ``modules`` ((name, module) pairs) that have forward hooks."""
    return [n for n, m in modules if isinstance(m, MultiheadAttention) and _hooked(m)]


def _attend(mha: nn.MultiheadAttention, query, key, value):
    """``_mha_core`` on 2-D operands, or the module call with [1, L, E] views when ``mha`` is hooked."""
    if not _hooked(mha):
        return _mha_core(mha, query, key, value)
    k = key.unsqueeze(0)
    out = mha(query=query.unsqueeze(0), key=k, value=k if value is key else value.unsqueeze(0))
    return _rows(out[0])


def _rows(t: torch.Tensor) -> torch.Tensor:
    assert t.dim() == 3 and t.shape[0] == 1, "the ModalTune path runs one slide per step (batch 1, train_modaltune.py:78)"
    return t.squeeze(0)   # a view both ways: the backward of t[0] zero-fills and copies a [1, L, 768] gradient


def _pos_rows(pos: Optional[torch.Tensor], rows: int) -> Optional[torch.Tensor]:
    if pos is None:
        return None
    p = pos.reshape(-1, pos.shape[-1])
    assert p.shape[0] == rows, "positional embedding must have one row per token"
    return p


class SelfAttentionLayer(nn.Module):
    """Prompt self-attention over the ~66 modal tokens (reference :18-99).  Negligible work: plain fp32 math."""

    def __init__(self, d_model, nheads, dropout=0.0, normalize_before=False, with_cffn=False, cffn_ratio=1.0):
        super().__init__()
        self.with_cffn = with_cffn
        self.cffn_ratio = cffn_ratio
        embed_model = d_model
        if self.with_cffn:
            embed_model = int(d_model * cffn_ratio)
            self.q_proj = nn.Linear(d_model, embed_model)
            self.output_proj = nn.Linear(embed_model, d_model)
        self.self_attn = MultiheadAttention(embed_model, nheads, dropout=dropout, batch_first=True, kdim=d_model,
                                            vdim=d_model)
        self.norm = nn.LayerNorm(d_model)
        self.dropout = nn.Dropout(dropout)
        self.normalize_before = normalize_before
        self._reset_parameters()

    def _reset_parameters(self):
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)

    def forward_pre(self, tgt, query_pos: Optional[torch.Tensor] = None):
        t = _rows(tgt).float()
        t2 = ops.layer_norm(t, self.norm.weight, self.norm.bias)
        qk = t2 if query_pos is None else t2 + _pos_rows(query_pos, t.shape[0]).to(t2.dtype)
        query = _lin(qk, self.q_proj.weight, self.q_proj.bias) if self.with_cffn else qk
        a = _attend(self.self_attn, query, qk, t2)
        if self.with_cffn:
            a = _lin(a, self.output_proj.weight, self.output_proj.bias)
        return (t + self.dropout(a)).unsqueeze(0)

    def forward(self, tgt, query_pos: Optional[torch.Tensor] = None):
        assert self.normalize_before, "ModalTune builds the prompt self-attention with normalize_before=True"
        return self.forward_pre(tgt, query_pos)


class CrossAttentionLayer(nn.Module):
    def __init__(self, d_model, nheads, dropout=0.0, normalize_before=False, with_cffn=False, cffn_ratio=1.0):
        super().__init__()
        self.with_cffn = with_cffn
        self.cffn_ratio = cffn_ratio
        embed_model = d_model
        if self.with_cffn:
            embed_model = int(d_model * cffn_ratio)
            self.q_proj = nn.Linear(d_model, embed_model)
            self.output_proj = nn.Linear(embed_model, d_model)
        self.multihead_attn = MultiheadAttention(embed_model, nheads, dropout=dropout, batch_first=True,
                                                 kdim=d_model, vdim=d_model)
        if normalize_before:
            self.norm_kq = nn.LayerNorm(d_model)
        self.norm = nn.LayerNorm(d_model)
        self.dropout = nn.Dropout(dropout)
        self.normalize_before = normalize_before
        self._reset_parameters()

    def _reset_parameters(self):
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)

    def attend(self, tgt, memory, pos=None, query_pos=None, tgt_row0: int = 0, mem_row0: int = 0):
        """The attention branch of ``forward_pre`` (:210-234) WITHOUT the trailing ``tgt +``: [Lq, 768] fp32.
        LayerNorm of both streams with the positional add fused; pos goes into the value input too.  ``*_row0`` = 1
        when the stream is the [cls | tiles] buffer and only the tile rows take part (no slice copies)."""
        assert self.multihead_attn.dropout == 0.0 or not self.training, "attention dropout is 0 in ModalTune's config"
        t2 = ops.layer_norm(tgt, self.norm.weight, self.norm.bias, add=_pos_rows(query_pos, tgt.shape[0] - tgt_row0),
                            row0=tgt_row0)
        mem = ops.layer_norm(memory, self.norm_kq.weight, self.norm_kq.bias,
                             add=_pos_rows(pos, memory.shape[0] - mem_row0), row0=mem_row0)
        query = _lin(t2, self.q_proj.weight, self.q_proj.bias) if self.with_cffn else t2
        a = _attend(self.multihead_attn, query, mem, mem)
        if self.with_cffn:
            a = _lin(a, self.output_proj.weight, self.output_proj.bias)
        return self.dropout(a)

    def forward_pre(self, tgt, memory, pos: Optional[torch.Tensor] = None, query_pos: Optional[torch.Tensor] = None):
        t = _rows(tgt).float()
        a = self.attend(t, _rows(memory).float(), pos, query_pos)
        return (t + a.float()).unsqueeze(0)

    def forward(self, tgt, memory, pos: Optional[torch.Tensor] = None, query_pos: Optional[torch.Tensor] = None):
        assert self.normalize_before, "ModalTune builds its cross-attention layers with normalize_before=True"
        return self.forward_pre(tgt, memory, pos, query_pos)


class FFNLayer(nn.Module):
    def __init__(self, d_model, dim_feedforward=256, dropout=0.0, normalize_before=False):
        super().__init__()
        self.linear1 = nn.Linear(d_model, dim_feedforward)
        self.dropout = nn.Dropout(dropout)
        self.linear2 = nn.Linear(dim_feedforward, d_model)
        self.norm = nn.LayerNorm(d_model)
        self.normalize_before = normalize_before
        self._reset_parameters()

    def _reset_parameters(self):
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)

    def forward_pre(self, tgt):
        t = _rows(tgt).float()
        h = ops.layer_norm(t, self.norm.weight, self.norm.bias)
        h = self.linear2(self.dropout(F.relu(self.linear1(h))))
        return h.unsqueeze(0)

    def forward(self, tgt, pos=None):
        assert self.normalize_before
        if pos is not None:
            tgt = tgt + pos
        return self.forward_pre(tgt)


class Extractor(nn.Module):
    """c <- c + (c + attn(c, x, query_pos=pe)); c <- c + DropPath(FFN(c))   (reference :296-335)."""

    def __init__(self, dim, num_heads=6, with_cffn=True, cffn_ratio=0.25, drop=0.0, drop_path=0.0, with_cp=False):
        super().__init__()
        self.attn = CrossAttentionLayer(d_model=dim, nheads=num_heads, normalize_before=True, with_cffn=with_cffn,
                                        cffn_ratio=cffn_ratio)
        self.with_cffn = with_cffn
        self.with_cp = with_cp  # activation checkpointing is off in ModalTune's config and not needed at 180 GB
        if with_cffn:
            self.ffn = FFNLayer(dim, int(dim * cffn_ratio), drop, True)
            self.drop_path = DropPath(drop_path) if drop_path > 0.0 else nn.Identity()

    def forward(self, query, feat, pos=None):
        attn = self.attn(query, feat, None, pos)
        query = query + attn
        if self.with_cffn:
            query = query + self.drop_path(self.ffn(query))
        return query

    def kv_weights(self):
        """The k | v projection of this extractor's memory with ``norm_kq`` folded in: LN(x) Wkv^T + b =
        xhat (Wkv diag gamma)^T + (Wkv beta + b) for xhat = normalise(x) (``ops.shared_kv_project``)."""
        cl = self.attn
        mha = cl.multihead_attn
        e = mha.embed_dim
        wkv = torch.cat([mha.k_proj_weight, mha.v_proj_weight], 0)
        return wkv * cl.norm_kq.weight[None, :], torch.addmv(mha.in_proj_bias[e:], wkv, cl.norm_kq.bias)

    def forward_full(self, query, xfull, pos=None, kv=None):
        """Same as ``forward`` with ``feat`` = the tile rows (1..) of the [1, N, 768] [cls | tiles] buffer ``xfull``.
        ``kv``: this extractor's k | v [L, 384] already projected (a column slice of a projection shared with the other
        extractors of the block); the memory LayerNorm and projection are skipped."""
        c = _rows(query).float()
        if kv is not None:
            cl = self.attn
            mha = cl.multihead_attn
            e = mha.embed_dim
            t2 = ops.layer_norm(c, cl.norm.weight, cl.norm.bias, add=_pos_rows(pos, c.shape[0]))
            qq = _lin(t2, cl.q_proj.weight, cl.q_proj.bias) if cl.with_cffn else t2
            o = ops.cross_attention_kv(_lin(qq, mha.q_proj_weight, mha.in_proj_bias[:e]), kv, mha.num_heads)
            a = _lin(o, mha.out_proj.weight, mha.out_proj.bias)
            if cl.with_cffn:
                a = _lin(a, cl.output_proj.weight, cl.output_proj.bias)
            a = cl.dropout(a)
        else:
            a = self.attn.attend(c, _rows(xfull), None, pos, mem_row0=1)
        query = (c + (c + a)).unsqueeze(0)
        if self.with_cffn:
            query = query + self.drop_path(self.ffn(query))
        return query


class Injector(nn.Module):
    """x <- x + gamma * (x + attn(x, c, pos=pe))   (reference :338-369), tail fused in one kernel."""

    def __init__(self, dim, num_heads=6, init_values=0.0, with_cp=False, with_cffn=True, cffn_ratio=0.25):
        super().__init__()
        self.with_cp = with_cp
        self.attn = CrossAttentionLayer(d_model=dim, nheads=num_heads, normalize_before=True, with_cffn=with_cffn,
                                        cffn_ratio=cffn_ratio)
        self.gamma = nn.Parameter(init_values * torch.ones((dim)), requires_grad=True)

    def forward(self, query, feat, pos=None):
        x = _rows(query).float()
        if self._can_fuse():
            return self._fused(x, feat, pos, 0).unsqueeze(0)
        a = self.attn.attend(x, _rows(feat).float(), pos, None)
        return ops.gated_residual(x, a, self.gamma).unsqueeze(0)

    def _fused(self, x, feat, pos, row0):
        """One autograd node for the [L, 768] side (``ops.InjectorFn``); the 66 modal tokens and the weight compositions
        stay ordinary autograd ops (they are weight-sized)."""
        cl = self.attn
        mha = cl.multihead_attn
        e = mha.embed_dim
        b = mha.in_proj_bias
        mem = _rows(feat).float()
        mem = ops.layer_norm(mem, cl.norm_kq.weight, cl.norm_kq.bias, add=_pos_rows(pos, mem.shape[0]))
        kv = _lin(mem, torch.cat([mha.k_proj_weight, mha.v_proj_weight], 0), b[e:])
        if cl.with_cffn:   # q = (t2 Wc^T + bc) Wm^T + bm  and  a = (o Wo^T + bo) Wout^T + bout as single maps
            wq = mha.q_proj_weight @ cl.q_proj.weight
            bq = torch.addmv(b[:e], mha.q_proj_weight, cl.q_proj.bias)
            wo = cl.output_proj.weight @ mha.out_proj.weight
            bo = torch.addmv(cl.output_proj.bias, cl.output_proj.weight, mha.out_proj.bias)
        else:
            wq, bq, wo, bo = mha.q_proj_weight, b[:e], mha.out_proj.weight, mha.out_proj.bias
        return ops.injector(x, kv, cl.norm.weight, cl.norm.bias, wq, bq, wo, bo, self.gamma, row0, mha.num_heads)

    def _can_fuse(self):
        cl = self.attn
        return (config.flag("injector_fused") and cl.normalize_before and not _hooked(cl.multihead_attn)
                and not (self.training and (cl.dropout.p > 0.0 or cl.multihead_attn.dropout > 0.0)))

    def forward_full(self, xfull, feat, pos=None):
        """Same as ``forward`` on the tile rows (1..) of the [1, N, 768] [cls | tiles] buffer; the cls row passes through."""
        x = _rows(xfull)
        if self._can_fuse():
            return self._fused(x, feat, pos, 1).unsqueeze(0)
        a = self.attn.attend(x, _rows(feat).float(), pos, None, tgt_row0=1)
        return ops.gated_residual(x, a, self.gamma, row0=1).unsqueeze(0)


class InteractionBlockWithCls(nn.Module):
    def __init__(self, dim, num_heads=6, drop=0.0, drop_path=0.0, with_cffn=True, cffn_ratio=0.25, init_values=0.0,
                 extra_extractor=False, with_cp=False):
        super().__init__()
        self.injector = Injector(dim=dim, num_heads=num_heads, init_values=init_values, with_cp=with_cp,
                                 with_cffn=with_cffn, cffn_ratio=cffn_ratio)
        self.extractor = Extractor(dim=dim, num_heads=num_heads, with_cffn=with_cffn, cffn_ratio=cffn_ratio,
                                   drop=drop, drop_path=drop_path, with_cp=with_cp)
        if extra_extractor:
            self.extra_extractors = nn.Sequential(*[
                Extractor(dim=dim, num_heads=num_heads, with_cffn=with_cffn, cffn_ratio=cffn_ratio, drop=drop,
                          drop_path=drop_path, with_cp=with_cp) for _ in range(2)])
        else:
            self.extra_extractors = None


class InteractionBlockWithCls_LongNetViT(InteractionBlockWithCls):
    """Injector -> [cls | x] through the frozen LongNet layers -> Extractor(s)   (reference :459-523)."""

    def forward(self, x, c, cls, blocks, incremental_state, layer_configs, query_pos=None):
        x = self.injector(query=x, feat=c, pos=query_pos)
        x = torch.cat((cls, x), dim=1)
        for idx, blk in enumerate(blocks):
            x, _ = blk(x, incremental_state=(incremental_state[idx] if incremental_state is not None else None),
                       **layer_configs)
        cls, x = x[:, :1], x[:, 1:]
        c = self.extractor(query=c, feat=x, pos=query_pos)
        if self.extra_extractors is not None:
            for extractor in self.extra_extractors:
                c = extractor(query=c, feat=x, pos=query_pos)
        return x, c, cls

    def forward_full(self, xfull, c, blocks, incremental_state, layer_configs, query_pos=None):
        """``forward`` on the [1, N, 768] buffer that keeps cls at row 0: the reference's ``cat((cls, x))`` and
        ``x[:, :1], x[:, 1:]`` (:492-505) and their backward copies disappear; same arithmetic."""
        xfull = self.injector.forward_full(xfull, c, query_pos)
        for idx, blk in enumerate(blocks):
            xfull, _ = blk(xfull, incremental_state=(incremental_state[idx] if incremental_state is not None else None),
                           **layer_configs)
        exts = [self.extractor, *(self.extra_extractors or ())]
        if (self.extra_extractors is not None and config.shared_extractor_kv()
                and not any(_hooked(e.attn.multihead_attn) for e in exts)):
            # the three extractors of the last block read the same slide tokens: one normalisation pass and one GEMM
            # for all their k | v projections (ops.SharedKVProjectFn), each then attends on its column slice.  A hooked
            # extractor needs its own attention call: then every extractor of the block projects for itself
            wb = [e.kv_weights() for e in exts]
            kv_all = ops.shared_kv_project(_rows(xfull), torch.cat([w for w, _ in wb], 0), torch.cat([b for _, b in wb], 0), 1)
            for e, kv in zip(exts, torch.split(kv_all, kv_all.shape[1] // len(exts), dim=1)):
                c = e.forward_full(c, xfull, query_pos, kv=kv)
            return xfull, c
        c = self.extractor.forward_full(c, xfull, query_pos)
        if self.extra_extractors is not None:
            for extractor in self.extra_extractors:
                c = extractor.forward_full(c, xfull, query_pos)
        return xfull, c
