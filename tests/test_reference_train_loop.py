"""Drop-in at the level of the reference's OWN training loop (SURVEY.md §8f rank 1, north-star "train_modaltune.py runs
unchanged"): ``MILTextGeneTrainer_multitask.init_model_and_optimizer / multitask_forward / train_one_epoch`` are executed
UNMODIFIED from ``/root/reference/train_modaltune.py`` (:118-243) and, for the pan-cancer variant with its 4-way task
one-hot, ``/root/reference/train_modaltune_pancancer.py`` (:41-134), once with the reference's model classes and once with
the B200 classes swapped in through the ``Aggregator`` registry exactly as INTEGRATION.md §2 shows.  Same seeded weights,
same synthetic cases, AdamW steps included: the epoch loss and the updated parameters must agree.

Only runs where the reference tree exists (the build container); nothing here travels to the GPU box.  On CPU the
kernel wrappers are the torch stand-ins of ``tests/cpu_kernels.py`` (test infrastructure), so what this pins is the
interface: constructor keywords, ``model(x=, coords=, genes=, clinical=, task_token=)``, ``is_multi``, the trainable /
frozen split the optimizer filter sees, train()/eval() switching, state-dict names.  The trainer object is built without
``Trainer.__init__`` (which needs the dataset files, wandb and an output directory -- all outside the hot path).
"""
import argparse
import os
import sys
import types

import pytest
import torch
from torch import nn

from modaltune_b200 import config, synthetic
from tests import cpu_kernels, helpers
from tests.golden import ref_shims

pytestmark = pytest.mark.skipif(not os.path.isdir(ref_shims.REFERENCE_ROOT),
                                reason="needs a checkout of the original ModalTune project: set MODALTUNE_REFERENCE to it")

L_TILES, N_CASES = 200, 2


class _WarmupScheduler:
    """warmup_scheduler.GradualWarmupScheduler is not installed: the loop only calls ``.step()`` once per epoch."""

    def __init__(self, optimizer, multiplier, total_epoch, after_scheduler=None):
        self.optimizer, self.multiplier, self.total_epoch, self.after, self.epoch = optimizer, multiplier, total_epoch, after_scheduler, 0
        self.base = [g["lr"] for g in optimizer.param_groups]

    def step(self):
        self.epoch += 1
        for g, b in zip(self.optimizer.param_groups, self.base):
            g["lr"] = b * ((self.multiplier - 1.0) * min(self.epoch, self.total_epoch) / self.total_epoch + 1.0)


SCRIPTS = {   # script -> (trainer class, --num_tasks default of that script)
    "train_modaltune": ("MILTextGeneTrainer_multitask", 3),
    "train_modaltune_pancancer": ("MILTextGeneTrainer_multitask_PC", 4),
}


def _import_reference_script(script):
    ref_shims.install()
    if "wandb" not in sys.modules:
        try:
            import wandb  # noqa: F401
        except Exception:
            sys.modules["wandb"] = types.ModuleType("wandb")
    import importlib

    tm = importlib.import_module(script)   # the untouched script: /root/reference/<script>.py
    import train_modaltune                 # the pan-cancer trainer inherits init_model_and_optimizer from this module

    train_modaltune.GradualWarmupScheduler = _WarmupScheduler
    return tm


def _make_trainer(tm, script, groups):
    import json

    cls_name, num_tasks = SCRIPTS[script]
    tr = object.__new__(getattr(tm, cls_name))              # skip Trainer.__init__ (datasets, wandb, output dirs)
    tr.args = argparse.Namespace(mil_name="longnetvit_gene_clinical_adapter", num_tasks=num_tasks, lr=2e-4, weight_decay=1e-2,
                                 beta1=0.9, beta2=0.999, num_epochs=20, world_size=1, use_amp=False, eval_interval=1000)
    tr.device = "cpu"
    with open(os.path.join(ref_shims.REFERENCE_ROOT, "model_configs", "modaltune_gigapath_config.json")) as f:
        tr.model_config = json.load(f)
    tr.gene_group_defination = groups
    tr.loss_fn = nn.KLDivLoss(reduction="sum")
    tr.temperature = 1.0
    tr.scaler = torch.amp.GradScaler("cpu", enabled=False)
    import train_modaltune

    tr.projector = train_modaltune.Projection_layer(input_dim=512, out_dim=tr.model_config["output_dim"])
    tr.projector.load_state_dict(synthetic.seeded_projector_state(0))
    tr.current_epoch = 1                                    # 1 % eval_interval != 0: no probe evaluation
    return tr


def _cases():
    out = []
    for i in range(N_CASES):
        s = synthetic.synthetic_slide(L_TILES, seed=900 + i, group_sizes=helpers.SMALL_GROUPS)
        # the tuple FeaturesGeneTextDataset yields through a batch-1 DataLoader (data_utils/datasets.py:180-285)
        out.append((s["x"], s["coords"], s["text"].unsqueeze(0), s["clinical"], s["genes"], torch.zeros(1), [f"case{i}"]))
    return out


def _write_synthetic_dataset(root, n_cases=N_CASES, n_tiles=L_TILES):
    """The on-disk inputs of the reference's FeaturesGeneTextDataset (data_utils/datasets.py:144-285), synthetic:
    feature bags ``{"features": [n, 1536], "coords": [n, 2]}``, the text-embedding dict ``{case_id: [4, 512]}``, the
    clinical dict ``{case_id: [5]}``, a genomics csv with the 4 987 pathway genes, and the datalist of the json splits."""
    import pandas as pd

    genes = pd.read_csv(os.path.join(ref_shims.REFERENCE_ROOT, "dataset", "gene_pathway_processed_v2.csv"))["gene"].tolist()
    g = torch.Generator().manual_seed(77)
    datalist, text, clin, rows = [], {}, {}, []
    for i in range(n_cases):
        cid = f"TCGA-XX-{i:04d}"
        s = synthetic.synthetic_slide(n_tiles, seed=700 + i, group_sizes=[1])
        path = os.path.join(root, f"{cid}.pt")
        torch.save({"features": s["x"][0].clone(), "coords": s["coords"][0].clone()}, path)
        datalist.append({"case_id": cid, "case_submitter_id": cid, "features_path": path, "primary_class": i % 2})
        text[cid] = torch.randn(4, 512, generator=g)
        clin[cid] = torch.randn(5, generator=g)
        rows.append([cid] + torch.randn(len(genes), generator=g).tolist())
    csv = os.path.join(root, "genomics.csv")
    pd.DataFrame(rows, columns=["case_id"] + genes).to_csv(csv, index=False)
    torch.save(text, os.path.join(root, "text.pt"))
    torch.save(clin, os.path.join(root, "clinical.pt"))
    return datalist, csv


def test_reference_dataset_and_loader_feed_the_b200_modules(tmp_path):
    """Files -> the reference's FeaturesGeneTextDataset -> the reference's ``Trainer.get_train_iterator`` DataLoader ->
    the reference's ``train_one_epoch`` -> B200 module classes (331 pathway groups of the real pathway table)."""
    from functools import partial

    tm = _import_reference_script("train_modaltune")
    from data_utils.datasets import FeaturesGeneTextDataset
    from models.aggregators import Aggregator as RefAggregator
    from models.genomic_utils.define_gene_groups import pathway_gene_groups
    from modaltune_b200.longvit_adapter import Aggregator as B200Aggregator
    import pandas as pd

    datalist, csv = _write_synthetic_dataset(str(tmp_path))
    groups = pathway_gene_groups(gene_df=pd.read_csv(csv), group_definations=True)    # train_modaltune.py:93-95
    assert len(groups) == 331
    saved = dict(RefAggregator.subclasses)
    try:
        RefAggregator.subclasses.update(B200Aggregator.subclasses)
        tr = _make_trainer(tm, "train_modaltune", groups)
        tr.args.__dict__.update(labelset="primary_class", text_location=os.path.join(str(tmp_path), "text.pt"),
                                genomics_csv_path=csv, clinical_location=os.path.join(str(tmp_path), "clinical.pt"),
                                batch_size=1, drop_last=False, workers=0)
        tr.train_transforms = None
        tr.Dataset_Class = partial(FeaturesGeneTextDataset, case_wise=True, return_case=True,          # :98-103
                                   gene_group_defination=groups, threshold=25000)
        torch.manual_seed(0)
        with cpu_kernels.installed():
            tr.init_model_and_optimizer()
            loader = tm.Trainer.get_train_iterator(tr, datalist)                                   # base_trainer.py:278-300
            tr.model.eval()
            tr.model.train = lambda mode=True: tr.model
            w0 = tr.model.interactions[0].injector.gamma.detach().clone()
            with config.using(mode="fp32"):
                loss = tr.train_one_epoch(loader)[3]
    finally:
        RefAggregator.subclasses.clear()
        RefAggregator.subclasses.update(saved)
    assert len(loader) == N_CASES and loss == loss and 0.0 < loss < 100.0
    assert not torch.equal(w0, tr.model.interactions[0].injector.gamma.detach())    # the optimizer stepped our parameters


def _run_epoch(tm, script, swap: bool):
    from models.aggregators import Aggregator as RefAggregator
    from modaltune_b200.longvit_adapter import Aggregator as B200Aggregator

    groups = {i: ["g"] * n for i, n in enumerate(helpers.SMALL_GROUPS)}
    saved = dict(RefAggregator.subclasses)
    try:
        if swap:
            RefAggregator.subclasses.update(B200Aggregator.subclasses)   # INTEGRATION.md §2: the whole integration
        tr = _make_trainer(tm, script, groups)
        torch.manual_seed(0)
        tr.init_model_and_optimizer()                       # reference code: Aggregator.create(...) + AdamW + schedulers
    finally:
        RefAggregator.subclasses.clear()
        RefAggregator.subclasses.update(saved)
    synthetic.seeded_init_(tr.model.named_parameters(), seed=0)
    # dropout / drop-path / AlphaDropout are stochastic and cannot be bit-matched between two implementations:
    # keep the loop's ``self.model.train()`` call but make it leave the modules in eval mode (parity is defined there)
    tr.model.eval()
    tr.model.train = lambda mode=True: tr.model
    before = {k: p.detach().clone() for k, p in tr.model.named_parameters() if p.requires_grad}
    with config.using(mode="fp32"):
        loss = tr.train_one_epoch(_cases())[3]              # reference code: forward x3, KL loss, backward, AdamW step
    after = {k: p.detach().clone() for k, p in tr.model.named_parameters() if p.requires_grad}
    return tr, float(loss), before, after


@pytest.mark.parametrize("script", sorted(SCRIPTS))
def test_reference_training_loop_runs_the_b200_modules_unchanged(script):
    tm = _import_reference_script(script)
    ref_tr, ref_loss, ref_before, ref_after = _run_epoch(tm, script, swap=False)
    with cpu_kernels.installed():
        our_tr, our_loss, our_before, our_after = _run_epoch(tm, script, swap=True)
    import modaltune_b200.longvit_adapter as ours

    assert type(our_tr.model) is ours.LongNetGeneSimpleClinicalAdapter and type(ref_tr.model) is not type(our_tr.model)
    assert our_tr.model.is_multi and set(our_before) == set(ref_before)          # same trainable set for the optimizer
    assert abs(our_loss - ref_loss) <= 1e-4 * abs(ref_loss), (our_loss, ref_loss)
    # AdamW's first steps are sign-like (update = -lr * m / (sqrt(v) + eps)): an element whose gradient is numerical noise
    # around an analytic zero (e.g. a bias feeding a LayerNorm) gets a random +-lr in BOTH implementations, so the
    # per-tensor comparison is made on the well-conditioned tensors and the noise-only ones are bounded in number.
    cosines, num, den_r, den_o = {}, 0.0, 0.0, 0.0
    for k in ref_before:
        assert torch.equal(our_before[k], ref_before[k]), k
        d_ref = (ref_after[k] - ref_before[k]).flatten().double()
        d_our = (our_after[k] - our_before[k]).flatten().double()
        if float(d_ref.abs().max()) == 0.0:
            assert float(d_our.abs().max()) == 0.0, k        # parameters without gradient stay put in both
            continue
        num += float(torch.dot(d_ref, d_our))
        den_r += float(d_ref.square().sum())
        den_o += float(d_our.square().sum())
        cosines[k] = float(torch.dot(d_ref, d_our) / (d_ref.norm() * d_our.norm() + 1e-30))
    assert len(cosines) > 100
    assert num / (den_r ** 0.5 * den_o ** 0.5) > 0.99, num / (den_r ** 0.5 * den_o ** 0.5)
    good = sum(c > 0.99 for c in cosines.values())
    assert good >= 0.95 * len(cosines), sorted(cosines.items(), key=lambda kv: kv[1])[:10]
