"""SURVEY.md 8(f1): the reference's ``train_modaltune.py`` runs BYTE-UNCHANGED, end to end (its argparse,
``Trainer.__init__``, dataset files -> ``FeaturesGeneTextDataset`` -> DataLoader, ``run()``: training epoch, probe
evaluation, validation, checkpoint, test), through ``python -m modaltune_b200.launcher`` with the B200 module classes
swapped in -- and lands where the same script lands with the reference's own classes.

* CPU (build container, reference at /root/reference): in-process, kernel wrappers replaced by the torch stand-ins of
  ``tests/cpu_kernels.py``; both runs in fp32.
* GPU (``-m gpu``, reference staged under oracle/_ref/reference by ``__graft_entry__.build()``): two subprocesses on
  the B200 -- ours in bf16 mode against the reference's real GPU path (fp16 autocast + flash-attn), the same-box
  end-to-end comparison of BASELINE.md 4.
"""
import contextlib
import glob
import io
import os
import re
import subprocess
import sys

import pytest
import torch

from modaltune_b200 import launcher
from tests import cpu_kernels

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPT_ARGS = ["--mil_name", "longnetvit_gene_clinical_adapter", "--model_config", "modaltune_gigapath_config",
               "--num_epochs", "1", "--num_folds", "1", "--workers", "0", "--eval_interval", "1", "--num_classes", "2",
               "--lr", "0.0002"]


def _reference_or_skip():
    try:
        staged = os.path.join(ROOT, "oracle", "_ref", "reference")   # test infrastructure: staged by build()
        return launcher.find_reference(staged if os.path.isdir(staged) and not os.path.isdir("/root/reference") else None)
    except FileNotFoundError:
        pytest.skip("needs a checkout of the original ModalTune project: set MODALTUNE_REFERENCE to it")


def _losses(text):
    return [float(v) for v in re.findall(r"train_cls_loss: ([0-9.eE+-]+)", text)], \
           [float(v) for v in re.findall(r"Validation loss: ([0-9.eE+-]+)", text)]


def test_train_script_unchanged_end_to_end_cpu(tmp_path):
    ref = _reference_or_skip()
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import ref_shims

    launcher.install_shims(ref)  # the launcher's own stand-ins first (working warm-up scheduler, Cox stand-in) ...
    ref_shims.install()          # ... then the plain-math flash_attn_func the reference lacks on CPU (test infrastructure)
    out = {}
    for classes in ("ours", "reference"):
        data = str(tmp_path / classes)
        buf = io.StringIO()
        ctx = cpu_kernels.installed() if classes == "ours" else contextlib.nullcontext()
        with ctx, contextlib.redirect_stdout(buf):
            launcher.main(["--reference", ref, "--classes", classes, "--synthetic", data, "--cases", "2", "--tiles", "48",
                           "--seeded-init", "0", "--deterministic", "--device", "cpu", "--mode", "fp32",
                           "train_modaltune.py", *SCRIPT_ARGS])
        text = buf.getvalue()
        weights = glob.glob(os.path.join(data, "results", "*", "best_model_weights.pt"))
        assert len(weights) == 1, text[-2000:]
        out[classes] = (_losses(text), torch.load(weights[0]), text)
        assert "test key metric of" in text                      # the script ran to the end of Trainer.run()
    (tr_o, va_o), sd_o, _ = out["ours"]
    (tr_r, va_r), sd_r, _ = out["reference"]
    assert len(tr_o) == 1 and len(va_o) >= 2 and len(tr_r) == 1
    assert abs(tr_o[0] - tr_r[0]) <= 1e-3 * abs(tr_r[0]), (tr_o, tr_r)
    assert abs(va_o[0] - va_r[0]) <= 5e-2 * abs(va_r[0]), (va_o, va_r)   # after two AdamW steps (sign-like updates)
    assert set(sd_o) | {"pos_embed"} == set(sd_r) | {"pos_embed"}          # checkpoints name the same tensors
    moved = sum(not torch.equal(sd_o[k], sd_r[k]) for k in sd_o if k in sd_r)
    assert moved > 100                                                       # the optimizer stepped (Adam noise differs)


@pytest.mark.gpu
def test_train_script_unchanged_end_to_end_b200(tmp_path):
    ref = _reference_or_skip()
    out = {}
    for classes, extra_launcher, extra_script in (("ours", ["--mode", "bf16"], []), ("reference", [], ["--use_amp"])):
        data = str(tmp_path / classes)
        cmd = [sys.executable, "-m", "modaltune_b200.launcher", "--reference", ref, "--classes", classes, "--synthetic", data,
               "--cases", "3", "--tiles", "2500", "--seeded-init", "0", "--deterministic", "--device", "0", *extra_launcher,
               "train_modaltune.py", *SCRIPT_ARGS, *extra_script]
        r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (classes, r.stdout[-1500:], r.stderr[-3000:])
        assert "test key metric of" in r.stdout, r.stdout[-1500:]
        assert len(glob.glob(os.path.join(data, "results", "*", "best_model_weights.pt"))) == 1
        out[classes] = _losses(r.stdout)
    (tr_o, va_o), (tr_r, va_r) = out["ours"], out["reference"]
    assert len(tr_o) == 1 and len(tr_r) == 1 and len(va_o) >= 1 and len(va_r) >= 1
    # bf16-mode tolerance of BASELINE.json (2e-2) on the epoch loss; the reference side is its own fp16 autocast path
    assert abs(tr_o[0] - tr_r[0]) <= 2e-2 * abs(tr_r[0]), (tr_o, tr_r)
