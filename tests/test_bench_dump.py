"""``bench.py --dump-outputs``: the files written for the last timed step.  On CPU the writer, with the kernel
stand-ins of ``tests/cpu_kernels.py``; on the GPU the whole benchmark run, twice."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from modaltune_b200 import config, synthetic, train_step
from tests import cpu_kernels, helpers


def test_dump_outputs_writes_what_the_step_returned(tmp_path, monkeypatch):
    model = helpers.build_model(helpers.SMALL_GROUPS)
    proj = helpers.build_projector(0)
    slide = synthetic.synthetic_slide(64, seed=3, group_sizes=helpers.SMALL_GROUPS)
    with cpu_kernels.installed(), config.using(mode="fp32"):
        loss, logits = train_step.forward_backward(model, proj, slide)
    params = [p for p in model.parameters() if p.requires_grad]
    flat = torch.cat([p.grad.reshape(-1) for p in params]).numpy()
    assert flat.size > bench.DUMP_GRAD_SAMPLE          # the sampled case, as with the full model

    def dump(name):
        d = tmp_path / name
        bench.dump_outputs(str(d), loss, logits, params)
        return {f[:-len(".npy")]: np.load(d / f) for f in os.listdir(d)}, sum(f.stat().st_size for f in d.iterdir())

    out, size = dump("a")
    assert set(out) == {"loss", "logits", "grad_norms", "grad_sample"}
    assert size <= 64 << 20
    assert out["loss"].dtype == np.float32 and out["loss"] == np.float32(float(loss))
    assert out["logits"].dtype == np.float32 and np.array_equal(out["logits"], logits.numpy())
    norms = np.array([float(p.grad.double().norm()) for p in params])
    assert out["grad_norms"].dtype == np.float64 and np.allclose(out["grad_norms"], norms, rtol=1e-12, atol=0)
    sample = out["grad_sample"]
    assert sample.dtype == np.float32 and sample.size == bench.DUMP_GRAD_SAMPLE and np.isin(sample, flat).all()
    again, _ = dump("b")                               # a fixed sample: two runs are comparable element by element
    assert all(np.array_equal(out[k], again[k]) for k in out)

    monkeypatch.setattr(bench, "DUMP_GRAD_SAMPLE", flat.size + 1)
    whole, _ = dump("c")                               # shorter than the sample: all of it, in parameter order
    assert np.array_equal(whole["grad_sample"], flat)


def _bench_dump(out_dir, steps):
    cmd = [sys.executable, "bench.py", "--tiles", "2000", "--steps", str(steps), "--warmup", "0", "--no-extras",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, cwd=os.path.dirname(os.path.abspath(bench.__file__)), capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    return line, {f[:-len(".npy")]: np.load(out_dir / f) for f in os.listdir(out_dir)}


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step_reproducibly(tmp_path):
    """The timed steps alternate between two seeded slides, so 2 and 4 steps end on the same slide and 3 on the other:
    the first two runs write the same files, the third a different loss.  Each dumped loss equals the loss the run reads
    back for that slide in its end-to-end region."""
    line2, a = _bench_dump(tmp_path / "a", 2)
    line4, b = _bench_dump(tmp_path / "b", 4)
    line3, c = _bench_dump(tmp_path / "c", 3)
    assert (line2["steps"], line4["steps"], line3["steps"]) == (2, 4, 3)
    for line, d in ((line2, a), (line4, b), (line3, c)):
        assert set(d) == {"loss", "logits", "grad_norms", "grad_sample"}
        assert all(np.isfinite(v).all() for v in d.values())
        assert abs(float(d["loss"]) - line["loss"]) <= 1e-6 * abs(line["loss"])
    assert float(a["loss"]) == pytest.approx(float(b["loss"]), rel=1e-6)
    assert float(c["loss"]) != pytest.approx(float(b["loss"]), rel=1e-3)
    assert np.allclose(a["logits"], b["logits"], rtol=1e-5, atol=1e-6 * np.abs(b["logits"]).max())
    # gradients: atomic accumulation order varies between runs, so equal up to rounding
    assert np.allclose(a["grad_norms"], b["grad_norms"], rtol=1e-3, atol=1e-4 * b["grad_norms"].max())
    assert np.abs(a["grad_sample"] - b["grad_sample"]).max() <= 1e-3 * np.abs(b["grad_sample"]).max()
