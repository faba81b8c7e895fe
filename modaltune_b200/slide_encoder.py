"""Drop-in ``LongNetViT`` (Prov-GigaPath slide encoder) running on the modaltune_b200 kernels.

Mirrors the interface of the reference class ``models/prov_gigapath/gigapath/slide_encoder.py:59-322`` that the Modal
Adapter touches: constructor keywords from the model JSON, attributes ``patch_embed``, ``cls_token``, ``pos_embed``
(see below), ``coords_to_pos``, ``encoder.prepare_forward``, ``encoder.layers[i](x, incremental_state=None, rel_pos=...,
encoder_padding_mask=..., attn_mask=..., multiway_split_position=...) -> (x, None)``, ``depth``, ``embed_dim``,
``drop_path_rate``, ``global_pool``, ``load_slide_encoder`` and ``forward(x, coords, all_layer_embed=False)``.
Parameter names and shapes equal the reference's, so ``slide_encoder.pth`` and ModalTune checkpoints load unchanged
(SURVEY.md §8b).  The submodules only HOLD the parameters: the arithmetic of a layer is one fused autograd node
(``ops.FrozenEncoderLayerFn``) over hand-written kernels + cuBLAS GEMMs.

Differences by design:
* ``pos_embed`` is not materialised as the reference's [1, 1_000_001, 768] fp32 buffer (3 GB, ``slide_encoder.py:118``).
  The 2-D sincos table is separable (``pos_embed.py:34-81``): ``pos_embed[1 + i*G + j] = [T[j] | T[i]]`` with one
  [G, 384] factor ``pos_table``; the embedding kernel adds it on the fly.  ``pos_embed_rows(pos)`` reproduces any rows.
* in ``train()`` mode the frozen encoder applies its Dropout(0.25) / DropPath like the reference (encoder.py:149-152,
  169-170, 339; feedforward_network.py:142), fused into the residual kernels with counter-based masks that the backward
  regenerates; parity against the reference is defined in ``eval()`` mode (masks cannot be bit-matched), see DESIGN.md.
"""
from __future__ import annotations

import os
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from . import config, ops

DILATED_RATIO = (1, 2, 4, 8, 16)


def optimal_segment_lengths(max_wsi_size: int = 262144, tile_size: int = 256) -> List[int]:
    """``LongNetViT.get_optimal_segment_length`` (slide_encoder.py:163-182) -> [1024, 5792, 32768, 185363, 1048576]."""
    max_seq_len = (max_wsi_size // tile_size) ** 2
    seg = np.linspace(np.log2(1024), int(np.log2(max_seq_len)), 5)
    return [int(v) for v in np.power(2, seg).astype(int)]


def sincos_factor(ngrids: int, dim: int) -> torch.Tensor:
    """The 1-D factor T [ngrids, dim/2] of the 2-D sincos table, float64 math then fp32 (pos_embed.py:63-81)."""
    quarter = dim // 4
    omega = 1.0 / 10000 ** (np.arange(quarter, dtype=np.float64) / quarter)
    out = np.einsum("m,d->md", np.arange(ngrids, dtype=np.float64), omega)
    return torch.from_numpy(np.concatenate([np.sin(out), np.cos(out)], axis=1)).float()


class PatchEmbed(nn.Module):
    """slide_encoder.py:37-56 -- Linear(in_chans, embed_dim); the bias is added by the embedding kernel."""

    def __init__(self, in_chans: int = 1536, embed_dim: int = 768, norm_layer=None, bias: bool = True):
        super().__init__()
        self.proj = nn.Linear(in_chans, embed_dim, bias=bias)
        self.norm = norm_layer(embed_dim) if norm_layer else nn.Identity()

    def forward(self, x):
        return self.norm(self.proj(x))


class _SelfAttention(nn.Module):
    """Parameter holder with the names of torchscale's MultiheadAttention / DilatedAttention
    (TS/component/multihead_attention.py:22-54)."""

    def __init__(self, embed_dim: int, num_heads: int, eps: float):
        super().__init__()
        self.embed_dim, self.num_heads, self.head_dim = embed_dim, num_heads, embed_dim // num_heads
        self.k_proj = nn.Linear(embed_dim, embed_dim, bias=True)
        self.v_proj = nn.Linear(embed_dim, embed_dim, bias=True)
        self.q_proj = nn.Linear(embed_dim, embed_dim, bias=True)
        self.out_proj = nn.Linear(embed_dim, embed_dim, bias=True)
        self.inner_attn_ln = nn.LayerNorm(embed_dim, eps=eps)


class _FeedForward(nn.Module):
    """Parameter holder with the names of TS/component/feedforward_network.py:93-131."""

    def __init__(self, embed_dim: int, ffn_dim: int, eps: float):
        super().__init__()
        self.fc1 = nn.Linear(embed_dim, ffn_dim)
        self.fc2 = nn.Linear(ffn_dim, embed_dim)
        self.ffn_layernorm = nn.LayerNorm(ffn_dim, eps=eps)


class LongNetEncoderLayer(nn.Module):
    """One pre-LN / sub-LN LongNet block (TS/architecture/encoder.py:24-175 with DilatedAttention)."""

    def __init__(self, embed_dim: int, num_heads: int, ffn_dim: int, segment_lengths, ratios, eps: float = 1e-5,
                 dropout: float = 0.0, drop_path: float = 0.0, layer_index: int = 0):
        super().__init__()
        self.embed_dim = embed_dim
        # train-mode stochastic ops of the frozen layer (encoder.py:69-75,149-152,169-170; feedforward_network.py:142)
        self.dropout, self.drop_path_prob, self.layer_index = float(dropout), float(drop_path), int(layer_index)
        self.self_attn = _SelfAttention(embed_dim, num_heads, eps)
        self.self_attn_layer_norm = nn.LayerNorm(embed_dim, eps=eps)
        self.ffn = _FeedForward(embed_dim, ffn_dim, eps)
        self.final_layer_norm = nn.LayerNorm(embed_dim, eps=eps)
        self.segment_lengths = [int(s) for s in segment_lengths]
        self.ratios = [int(r) for r in ratios]
        self._weights = ops.FrozenLayerWeights()

    def runs_batched(self, x) -> bool:
        """Does a [B, N, 768] input (B > 1) run as ONE batched forward (``ops.encoder_layer_forward_batch``) instead of B
        layer calls: when autograd records nothing, in eval mode, in bf16 mode with the tcgen05 GEMMs.  Each sequence then
        gets bitwise what its own call gives it."""
        return (x.shape[0] > 1 and not (torch.is_grad_enabled() and x.requires_grad) and not self.training
                and ops.batched_forward_available())

    def forward(self, x, encoder_padding_mask=None, attn_mask=None, rel_pos=None, multiway_split_position=None,
                incremental_state=None):
        assert attn_mask is None and rel_pos is None and incremental_state is None, \
            "the LongNet slide encoder is called without masks / relative positions / incremental state"
        if any(p.requires_grad for p in self.parameters(recurse=True)):
            raise RuntimeError("modaltune_b200 runs the slide encoder frozen (longvit_adapter.py:78-80): its fused "
                               "backward produces input gradients only")
        B, N, E = x.shape
        cdt = config.compute_dtype()
        W = self._weights.refresh(self, cdt)
        geom = ops.Geometry.get(N, self.segment_lengths, self.ratios)
        impl = (config.attn_impl("fwd"), config.attn_impl("bwd"))
        rng = None
        if self.training and (self.dropout > 0.0 or self.drop_path_prob > 0.0):
            assert B == 1, "train-mode DropPath is drawn per sample; the ModalTune path runs one slide per step"
            rng = ops.train_rng(x.device, self.dropout, self.drop_path_prob, 2 * self.layer_index)
        if B == 1:   # pure views: the backward of x[0] would zero-fill and copy a [1, N, 768] gradient per layer
            return ops.frozen_encoder_layer(x.reshape(N, E).float(), W, geom, cdt, impl, rng).unsqueeze(0), None
        if self.runs_batched(x):
            y = ops.encoder_layer_forward_batch(x.reshape(B * N, E).float().contiguous(), W, geom, B, impl)
            return y.view(B, N, E), None
        outs = [ops.frozen_encoder_layer(x[b].float(), W, geom, cdt, impl, rng) for b in range(B)]
        y = torch.stack(outs, 0)
        return y, None


class LongNetEncoder(nn.Module):
    """``encoder`` attribute of LongNetViT (TS/architecture/encoder.py:178-436, TS/model/LongNet.py:53-82)."""

    def __init__(self, embed_dim: int, depth: int, num_heads: int, ffn_dim: int, segment_lengths, ratios,
                 eps: float = 1e-5, dropout: float = 0.0, drop_path_rate: float = 0.0):
        super().__init__()
        # DropPath probability grows linearly with depth (encoder.py:37-41: np.linspace(0, rate, layers)[depth])
        dp = [drop_path_rate * l / max(depth - 1, 1) for l in range(depth)] if drop_path_rate > 0 else [0.0] * depth
        self.layers = nn.ModuleList([
            LongNetEncoderLayer(embed_dim, num_heads, ffn_dim, segment_lengths, ratios, eps, dropout=dropout,
                                drop_path=dp[l], layer_index=l) for l in range(depth)])
        self.dropout = float(dropout)
        self.layer_norm = nn.LayerNorm(embed_dim, eps=eps)  # encoder_normalize_before; unused by the adapter
        self.embed_scale = 1.0  # no_scale_embedding=True
        self.num_layers = depth

    def prepare_forward(self, src_tokens, encoder_padding_mask=None, token_embeddings=None,
                        multiway_split_position=None, positions=None, **kwargs):
        """encoder.py:342-385: scale (1), dropout on the embedded tokens (:339, train mode only), mask multiply (ones)."""
        assert token_embeddings is not None, "the slide encoder is driven by token embeddings"
        emb = x = token_embeddings
        if self.training and self.dropout > 0.0:
            x = torch.nn.functional.dropout(emb, self.dropout, True)
        if encoder_padding_mask is None:
            encoder_padding_mask = torch.zeros(x.shape[:2], device=x.device, dtype=torch.bool)
        return x, emb, encoder_padding_mask, None

    def layer_forward(self, x, rel_pos_bias=None, encoder_padding_mask=None, attn_mask=None, return_all_hiddens=False,
                      multiway_split_position=None, features_only=False, incremental_state=None, **kwargs):
        states = [x] if return_all_hiddens else []
        for layer in self.layers:
            x, _ = layer(x, encoder_padding_mask=encoder_padding_mask, attn_mask=attn_mask, rel_pos=rel_pos_bias)
            if return_all_hiddens:
                states.append(x)
        x = torch.nn.functional.layer_norm(x, (x.shape[-1],), self.layer_norm.weight, self.layer_norm.bias,
                                           self.layer_norm.eps)
        return {"encoder_out": x, "encoder_padding_mask": encoder_padding_mask, "encoder_states": states,
                "l_aux": [None] * len(self.layers)}


class LongNetViT(nn.Module):
    def __init__(self, in_chans=1536, embed_dim=256, depth=12, slide_ngrids=1000, tile_size=256,
                 max_wsi_size=262144, norm_layer=None, global_pool=False, dropout=0.25, drop_path_rate=0.1,
                 return_feats=False, lora_adapter=False, lora_args=None, **kwargs):
        super().__init__()
        assert not lora_adapter, "LoRA dilated attention is not part of the ModalTune path (SURVEY.md §2 row 1)"
        self.depth = depth
        self.embed_dim = embed_dim
        self.drop_path_rate = drop_path_rate
        self.return_feats = return_feats
        self.tile_size = tile_size
        self.patch_embed = PatchEmbed(in_chans, embed_dim)
        self.slide_ngrids = slide_ngrids
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.register_buffer("pos_table", sincos_factor(slide_ngrids, embed_dim), persistent=False)
        self.encoder_name = "LongNet_{}_layers_{}_dim".format(depth, embed_dim)
        mlp_ratio = kwargs.get("mlp_ratio", 4.0)
        # LongNet_12_layers_768_dim: 16 heads (TS/model/LongNetConfig.py:166-179); dilation [1, 2, 4, 8, 16]
        assert embed_dim == ops.EMBED, "the kernels are built for the 768-d / 16-head GigaPath slide encoder"
        self.segment_lengths = optimal_segment_lengths(max_wsi_size, tile_size)
        self.encoder = LongNetEncoder(embed_dim, depth, ops.HEADS, int(embed_dim * mlp_ratio), self.segment_lengths,
                                      DILATED_RATIO, dropout=dropout, drop_path_rate=drop_path_rate)
        self.norm = nn.LayerNorm(embed_dim, eps=1e-6)  # unused by the adapter (longvit_adapter.py:309-312)
        self.global_pool = global_pool
        self.initialize_vit_weights()

    # -- initialisation (slide_encoder.py:144-196; sub-LN scaling TS/architecture/encoder.py:269-285) ------------------
    def initialize_vit_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.LayerNorm):
                nn.init.constant_(m.bias, 0)
                nn.init.constant_(m.weight, 1.0)
        nn.init.normal_(self.cls_token, std=0.02)

    def coords_to_pos(self, coords):
        c = torch.floor(coords / 256.0)
        return (c[..., 0] * self.slide_ngrids + c[..., 1]).long() + 1

    def pos_embed_rows(self, pos: torch.Tensor) -> torch.Tensor:
        """Rows of the reference's ``pos_embed`` table for indices ``pos`` (0 = cls row, all zeros)."""
        p = pos - 1
        i, j = torch.div(p, self.slide_ngrids, rounding_mode="floor"), p % self.slide_ngrids
        rows = torch.cat([self.pos_table[j.clamp(min=0)], self.pos_table[i.clamp(min=0)]], dim=-1)
        return torch.where((pos > 0).unsqueeze(-1), rows, torch.zeros_like(rows))

    def embed(self, x: torch.Tensor, coords: torch.Tensor) -> torch.Tensor:
        """PatchEmbed + positional embedding + cls row (A0): [B, L, C], [B, L, 2] -> [B, L+1, E] fp32."""
        cdt = config.compute_dtype()
        B, L, C = x.shape
        w = self.patch_embed.proj.weight
        if x.requires_grad or w.requires_grad:
            raise RuntimeError("the patch embedding is frozen and takes constant inputs on this path")
        outs = []
        with torch.no_grad():
            # fp32 operands; TF32 tensor-core GEMM in bf16 mode, exact fp32 in fp32 mode.  The token embedding feeds
            # every later op: rounding it to bf16 costs more gradient accuracy than all bf16 GEMMs of the encoder
            # together (DESIGN.md "numerics"), and the GEMM is 0.3% of the step's FLOPs.
            wq = w.detach().float()
            bias = self.patch_embed.proj.bias.detach().float().contiguous()
            cls = self.cls_token.detach().reshape(-1).float().contiguous()
            for b in range(B):
                if cdt == torch.float32:
                    proj = torch.matmul(x[b].float(), wq.t())
                else:
                    with ops._tf32():
                        proj = torch.matmul(x[b].float(), wq.t())
                # the reference divides by a literal 256.0 whatever ``tile_size`` says (slide_encoder.py:198-211);
                # ``coords_to_pos`` above and the kernel use the same divisor
                outs.append(ops.embed_assemble(proj, bias, coords[b].float().contiguous(), self.pos_table, cls, 256.0))
        return outs[0].unsqueeze(0) if B == 1 else torch.stack(outs, 0)

    def forward(self, x, coords, all_layer_embed=False):
        x = self.embed(x, coords)
        x, _, pad, rel = self.encoder.prepare_forward(src_tokens=None, token_embeddings=x)
        out = self.encoder.layer_forward(x=x, rel_pos_bias=rel, encoder_padding_mask=pad,
                                         return_all_hiddens=all_layer_embed)
        x_list = out["encoder_states"] if all_layer_embed else [out["encoder_out"]]
        outcomes = []
        for t in x_list:
            ln = lambda u: torch.nn.functional.layer_norm(u, (u.shape[-1],), self.norm.weight, self.norm.bias,
                                                          self.norm.eps)
            outcomes.append(ln(t[:, 1:, :].mean(dim=1)) if self.global_pool else ln(t)[:, 0])
        return (outcomes, x_list[-1]) if self.return_feats else outcomes

    def load_slide_encoder(self, pretrained=False, weights_location="./"):
        """slide_encoder.py:292-322: load ``slide_encoder.pth`` if present, else keep the random init."""
        if not pretrained:
            return None
        local_path = os.path.join(weights_location, "slide_encoder.pth")
        if os.path.exists(local_path):
            state_dict = torch.load(local_path, map_location="cpu")["model"]
            state_dict.pop("pos_embed", None)
            missing, unexpected = self.load_state_dict(state_dict, strict=False)
            for k in missing:
                print("Missing ", k)
            for k in unexpected:
                print("Unexpected ", k)
        else:
            print("Pretrained weights not found at {}. Randomly initialized the model!".format(local_path))
