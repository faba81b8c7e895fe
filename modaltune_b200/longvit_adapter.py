"""ModalTune-GigaPath model assembly on the modaltune_b200 kernels.

Drop-in for the reference's ``models/aggregators/longvit_adapter.py`` (``LongNetGeneAdapter`` :30-347,
``LongNetGeneSimpleClinicalAdapter`` :350-672) and its registry ``models/aggregators/aggregators.py:23-41``:
same registry names, constructor keywords (the model JSON is splatted into the constructor,
``train_modaltune.py:118-125``), forward signatures and parameter names, so checkpoints written by either side load
into the other (``tests/test_state_dict.py``).
"""
from __future__ import annotations

from typing import Any, Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import config
from .adapter_modules import (CrossAttentionLayer, Identity_mod, InteractionBlockWithCls_LongNetViT,
                              SelfAttentionLayer, recording_outputs)
from .gene_encoder import GeneEncoder_Group
from .slide_encoder import LongNetViT

# model_configs/other_configs.py:10-24 (hard-coded in the reference)
GENOMIC_CONFIG = {"latent_dim": 256, "depth": 3, "expansion_groups": 0.5, "expansion_dim": 0.5, "dropout": 0.25,
                  "cls_token": False, "n_classes": 2, "final_groups": 64}
# model_configs/modaltune_gigapath_config.json
GIGAPATH_CONFIG = {
    "in_chans": 1536, "embed_dim": 768, "depth": 12, "slide_ngrids": 1000, "tile_size": 256, "max_wsi_size": 262144,
    "global_pool": False, "dropout": 0.25, "drop_path_rate": 0.1, "mlp_ratio": 4,
    "num_heads": 12, "output_dim": 256, "init_values": 0.0, "geneclass_name": "gene_mixer_group",
    "interaction_indexes": [[0, 3], [4, 7], [8, 11]], "with_cffn": True, "cffn_ratio": 0.25,
    "add_prompt_feature": True, "use_extra_extractor": True, "freeze_vit": True, "with_cp": False,
    "use_prompt_sa": True, "prompt_dropout": 0.0, "prompt_agg": "avg", "token_agg": "sum", "pretrained": True,
    "clinfeat_dim": 5,
}
GIGAPATH_WEIGHT_LOC = "/huggingface/hub/models--prov-gigapath--prov-gigapath/"  # utils/constants.py:15


class Aggregator(nn.Module):
    """Name -> class registry (``Aggregator.register`` / ``Aggregator.create``, aggregators.py:23-41)."""

    subclasses: Dict[str, Any] = {}

    @classmethod
    def register(cls, subclass_name: str):
        def decorator(subclass: Any):
            cls.subclasses[subclass_name] = subclass
            return subclass
        return decorator

    @classmethod
    def create(cls, subclass_name: str, **params):
        if subclass_name not in cls.subclasses:
            raise ValueError("Unknown subclass name {}".format(subclass_name))
        return cls.subclasses[subclass_name](**params)


@Aggregator.register("longnetvit_gene_adapter")
class LongNetGeneAdapter(LongNetViT):
    """LongNet ViT with gene Modal Adapters and a task prompt."""

    _HAS_CLINICAL = False

    def __init__(self, num_heads=12, gene_group_defination={}, geneclass_name="gene_mixer_group", output_dim=256,
                 init_values=0.0, interaction_indexes=None, with_cffn=True, cffn_ratio=0.25, add_prompt_feature=True,
                 use_extra_extractor=True, freeze_vit=True, with_cp=False, use_prompt_sa=False, prompt_dropout=0.0,
                 prompt_agg="cls", token_agg="cat", pretrained=True, multi_task=1, clinfeat_dim=5, **kwargs):
        LongNetViT.__init__(self, **kwargs)
        self.load_slide_encoder(pretrained=pretrained, weights_location=GIGAPATH_WEIGHT_LOC)
        assert freeze_vit, "modaltune_b200 runs the slide encoder frozen (its fused backward is dX-only)"
        for _, param in self.named_parameters():
            param.requires_grad = False
        assert geneclass_name == "gene_mixer_group"
        self.mode = "feature"
        self.num_block = self.depth
        self.interaction_indexes = interaction_indexes
        self.add_prompt_feature = add_prompt_feature
        self.prompt_agg = prompt_agg
        self.token_agg = token_agg
        self.is_multi = multi_task > 1
        embed_dim = self.embed_dim
        n_int = len(interaction_indexes)
        self.interactions = nn.Sequential(*[
            InteractionBlockWithCls_LongNetViT(
                dim=embed_dim, num_heads=num_heads, init_values=init_values, drop_path=self.drop_path_rate,
                with_cffn=with_cffn, cffn_ratio=cffn_ratio,
                extra_extractor=(i == n_int - 1) and use_extra_extractor, with_cp=with_cp)
            for i in range(n_int)])
        self.prompt_selfattention = nn.Sequential(
            Identity_mod(),
            *[(SelfAttentionLayer(d_model=embed_dim, nheads=num_heads, dropout=prompt_dropout, normalize_before=True,
                                  with_cffn=with_cffn, cffn_ratio=cffn_ratio) if use_prompt_sa else Identity_mod())
              for _ in range(1, n_int)])
        self.gene_encoder = GeneEncoder_Group(**GENOMIC_CONFIG, output_dim=embed_dim, mode="feature",
                                              group_sizes=gene_group_defination,
                                              n_groups=len(gene_group_defination))
        num_gene_groups = self.gene_encoder.n_groups
        if self.prompt_agg == "cls":
            self.gene_cls = nn.Parameter(torch.zeros(1, 1, embed_dim))
            num_gene_groups += 1
            nn.init.trunc_normal_(self.gene_cls.data, std=0.02)
        n_lead = int(self.is_multi) + int(self._HAS_CLINICAL)
        self.gene_pe = nn.Parameter(torch.zeros(num_gene_groups + n_lead, embed_dim))
        if self.is_multi:
            self.task_weight = nn.Sequential(nn.Linear(multi_task, embed_dim), nn.LayerNorm(embed_dim))
            self.task_weight.apply(self._init_adapter_weights)
        if self._HAS_CLINICAL:
            self.clinical_mlp = nn.Sequential(nn.Linear(clinfeat_dim, embed_dim // 2), nn.ReLU(),
                                              nn.Linear(embed_dim // 2, embed_dim), nn.LayerNorm(embed_dim))
            self.clinical_mlp.apply(self._init_adapter_weights)
        n_cat = 2 + int(self.is_multi) + int(self._HAS_CLINICAL)
        if self.token_agg == "cat":
            self.final_norm = nn.LayerNorm(n_cat * embed_dim)
            self.final_project = nn.Linear(n_cat * embed_dim, output_dim)
        elif self.token_agg == "sum":
            self.final_norm = nn.LayerNorm(embed_dim)
            self.final_project = nn.Linear(embed_dim, output_dim)
        else:
            raise NotImplementedError
        # initialisation order of the reference (:176-182)
        self.interactions.apply(self._init_adapter_weights)
        for m in self.modules():
            if isinstance(m, (CrossAttentionLayer, SelfAttentionLayer)):
                m._reset_parameters()
        self.gene_encoder.apply(self._init_adapter_weights)
        self.final_project.apply(self._init_adapter_weights)
        self.final_norm.apply(self._init_adapter_weights)
        nn.init.trunc_normal_(self.gene_pe.data, std=0.02)

    @staticmethod
    def _init_adapter_weights(m):
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=0.02)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)

    # -- forward ---------------------------------------------------------------------------------------------------------
    def _shared_inputs(self, x, coords, genes):
        """The task-independent part of a forward: embedded slide tokens [1, N, 768] and the gene-encoder tokens."""
        return self.embed(x, coords), self.gene_encoder(genes)

    def forward_tasks(self, x, coords, genes, clinical=None, task_tokens=(), split_grads: bool = False):
        """Several task-conditioned passes over ONE slide (what ``multitask_forward`` does with one ``forward`` per task,
        train_modaltune.py:156-179).  The token embedding (frozen, deterministic: its dropout sits after it, in
        ``prepare_forward``) is computed once; the gene-encoder output is shared in eval mode and recomputed per pass in
        train mode, where the reference draws fresh dropout masks in every ``model(...)`` call.

        ``split_grads``: every pass reads the trainable parameters through its OWN leaf aliases (same storage, listed in
        ``self._pass_aliases`` for the caller, ``train_step.forward_backward``).  The autograd engine then delivers one
        gradient per (parameter, pass) instead of summing the passes' contributions with two tiny add kernels per
        parameter (~700 launches per step); the caller sums them with two multi-tensor adds."""
        emb = self.embed(x, coords)
        gene = None if self.training else self.gene_encoder(genes)
        self._pass_aliases = None
        if split_grads and config.flag("split_param_grads") and torch.is_grad_enabled() and len(task_tokens) > 1:
            # the gene encoder stays on the shared leaves: in eval mode it runs once for all passes, and in train mode its
            # 1 324 per-pathway gradients are strided slices of stacked tensors, which the multi-tensor add of
            # forward_backward would handle one tensor at a time (measured: +3.5 ms per train-mode step)
            named = [(n, p) for n, p in self.named_parameters() if p.requires_grad and not n.startswith("gene_encoder.")]
            self._pass_aliases = [{n: p.detach().requires_grad_(True) for n, p in named} for _ in task_tokens]

        def one_pass(t, k=0):
            if self._pass_aliases is not None:
                from torch.nn.utils.stateless import _reparametrize_module
                with _reparametrize_module(self, self._pass_aliases[k]):
                    shared = (emb, gene if gene is not None else self.gene_encoder(genes))
                    return self._adapter_forward(None, None, None, clinical, t, None, None, None, shared=shared)
            shared = (emb, gene if gene is not None else self.gene_encoder(genes))
            return self._adapter_forward(None, None, None, clinical, t, None, None, None, shared=shared)

        if not (config.pass_streams() and emb.is_cuda and len(task_tokens) > 1):
            return torch.cat([one_pass(t, k) for k, t in enumerate(task_tokens)], 0)
        # The task passes are independent until the loss: each one runs on its own CUDA stream (autograd replays the
        # backward of every node on the stream of its forward), so kernels of different passes overlap -- the tails of
        # the attention launches and the hundreds of tiny modal-token kernels fill each other's gaps.  Under CUDA-graph
        # capture the forks become parallel branches of the graph.
        cur = torch.cuda.current_stream()
        streams = self._task_streams(len(task_tokens) - 1)
        outs = [None] * len(task_tokens)
        hook_outputs = []   # what forward hooks on the attention modules received on the side streams
        gene_inputs = list(genes.values()) if isinstance(genes, dict) else list(genes)
        for k, t in enumerate(task_tokens):
            if k == 0:
                continue
            st = streams[k - 1]
            st.wait_stream(cur)
            # Everything allocated on the calling stream that this pass reads (forward AND backward, through autograd's
            # saved tensors) must be known to the allocator as in use on the side stream: otherwise its block can be
            # handed out again on the calling stream while a side-stream kernel is still queued to read it (seen as a
            # wrong task_weight gradient: the 12-byte one-hot task token was recycled during the backward).
            for tns in (emb, gene, clinical, t, *(gene_inputs if gene is None else ())):
                if torch.is_tensor(tns) and tns.is_cuda:
                    tns.record_stream(st)
            with torch.cuda.stream(st), recording_outputs(hook_outputs):
                outs[k] = one_pass(t, k)
        outs[0] = one_pass(task_tokens[0], 0)
        for k in range(1, len(task_tokens)):
            cur.wait_stream(streams[k - 1])
            outs[k].record_stream(cur)   # allocated on the side stream, read by the cat below on the calling stream
        for tns in hook_outputs:         # and these by the hook's owner after we return
            tns.record_stream(cur)
        return torch.cat(outs, 0)

    def join_pass_streams(self):
        """Make the current stream wait for everything queued on the task-pass streams (call after a backward)."""
        streams = self.__dict__.get("_streams", [])
        if not streams:
            return
        cur = torch.cuda.current_stream()
        for st in streams:
            cur.wait_stream(st)

    def _task_streams(self, n):
        pool = self.__dict__.setdefault("_streams", [])
        while len(pool) < n:
            pool.append(torch.cuda.Stream())
        return pool

    def _modal_tokens(self, gene_tokens, clinical, task_token):
        """[1, M, 768] modal tokens: (clinical) | (task) | (gene cls) | 64 pathway tokens  (:257-266, 568-584)."""
        c = gene_tokens
        if self.prompt_agg == "cls":
            c = torch.cat((self.gene_cls, c), dim=1)
        if self.is_multi:
            task_cls = self.task_weight(task_token.to(c.dtype).unsqueeze(0)).unsqueeze(0)
            c = torch.cat((task_cls, c), dim=1)
        if self._HAS_CLINICAL:
            c = torch.cat((self.clinical_mlp(clinical.to(c.dtype)).unsqueeze(0), c), dim=1)
        return c

    def _adapter_forward(self, x, coords, genes, clinical, task_token, attn_mask, multiway_split_position,
                         incremental_state, shared=None):
        if shared is None:
            shared = self._shared_inputs(x, coords, genes)
        x, gene_tokens = shared
        x, _, encoder_padding_mask, rel_pos_bias = self.encoder.prepare_forward(src_tokens=None, token_embeddings=x)
        layer_configs = {"rel_pos": rel_pos_bias,
                         "encoder_padding_mask": encoder_padding_mask if incremental_state is None else None,
                         "attn_mask": attn_mask, "multiway_split_position": multiway_split_position}
        c = self._modal_tokens(gene_tokens, clinical, task_token)
        for idx, blk in enumerate(self.encoder.layers[0:self.interaction_indexes[0][0]]):
            x, _ = blk(x, incremental_state=None, **layer_configs)
        # cls stays at row 0 of one [1, N, 768] buffer; Injector / Extractor work on rows 1.. in place
        for i, layer in enumerate(self.interactions):
            lo, hi = self.interaction_indexes[i][0], self.interaction_indexes[i][-1]
            c = self.prompt_selfattention[i](c, self.gene_pe)
            x, c = layer.forward_full(x, c, self.encoder.layers[lo:hi + 1], incremental_state, layer_configs,
                                      self.gene_pe)
        img_outcome = x[:, 1:].mean(dim=1).unsqueeze(0) if self.global_pool else x[:, :1]
        if self.add_prompt_feature:
            k = int(self._HAS_CLINICAL)
            m = int(self.is_multi)
            clinical_outcome = c[:, 0:k]
            task_outcome = c[:, k:k + m]
            if self.prompt_agg == "cls":
                gene_outcome = c[:, k + m:k + m + 1]
            elif self.prompt_agg == "avg":
                gene_outcome = c[:, k + m:].mean(dim=1).unsqueeze(1)
            else:
                raise NotImplementedError
            parts = [img_outcome] + ([task_outcome] if m else []) + [gene_outcome] + ([clinical_outcome] if k else [])
            if self.token_agg == "sum":
                outcome = parts[0]
                for p in parts[1:]:
                    outcome = outcome + p
            else:
                outcome = torch.cat(parts, dim=-1)
        else:
            outcome = img_outcome
        outcome = self.final_norm(outcome)
        return self.final_project(outcome.squeeze(1))

    def forward(self, x, coords, genes, task_token=None, attn_mask=None, multiway_split_position=None,
                incremental_state=None, **kwargs):
        return self._adapter_forward(x, coords, genes, None, task_token, attn_mask, multiway_split_position,
                                     incremental_state)


@Aggregator.register("longnetvit_gene_clinical_adapter")
class LongNetGeneSimpleClinicalAdapter(LongNetGeneAdapter):
    """LongNet ViT with gene Modal Adapters, a task prompt and clinical priors."""

    _HAS_CLINICAL = True

    def forward(self, x, coords, genes, clinical, task_token=None, attn_mask=None, multiway_split_position=None,
                incremental_state=None):
        return self._adapter_forward(x, coords, genes, clinical, task_token, attn_mask, multiway_split_position,
                                     incremental_state)
