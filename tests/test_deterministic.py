"""Host logic of deterministic mode (no GPU): how the switch resolves, what it selects, what it refuses, and that the
C ABI declares and exports the deterministic entry points."""
import ctypes
import os
import warnings

import pytest
import torch

from modaltune_b200 import _lib, config, ops, train_step

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(autouse=True)
def _restore():
    state = dict(config._state)
    flag, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    yield
    config._state.update(state)
    torch.use_deterministic_algorithms(flag, warn_only=warn)


def test_default_is_off_and_leaves_the_default_impls():
    if os.environ.get("MODALTUNE_B200_DETERMINISTIC", "0") not in ("", "0"):
        pytest.skip("the environment turns deterministic mode on")
    assert not config.deterministic()
    assert config.attn_impl("bwd") == config.AUTO_IMPL["bwd"] and config.attn_impl("fwd") == config.AUTO_IMPL["fwd"]


def test_switch_from_using_and_from_torch_flag():
    with config.using(deterministic=True):
        assert config.deterministic() and ops.dilated_bwd_impl(config.attn_impl("bwd")) == 4
        assert ops.dilated_bwd_impl(1) == 4 and ops.dilated_bwd_impl(4) == 4
        # what config reports stays the default selection: the forward is deterministic already
        assert config.attn_impl("bwd") == config.AUTO_IMPL["bwd"] and config.attn_impl("fwd") == config.AUTO_IMPL["fwd"]
    assert ops.dilated_bwd_impl(1) == 1 and ops.dilated_bwd_impl(2) == 2
    config.set_deterministic(False)
    torch.use_deterministic_algorithms(True)
    assert config.deterministic() and ops.dilated_bwd_impl(config.attn_impl("bwd")) == 4


def test_switch_from_the_environment():
    import subprocess
    import sys
    code = "from modaltune_b200 import config, ops; print(config.deterministic(), ops.dilated_bwd_impl(config.attn_impl('bwd')))"
    for val, want in (("1", "True 4"), ("0", f"False {config.AUTO_IMPL['bwd']}")):
        env = dict(os.environ, MODALTUNE_B200_DETERMINISTIC=val, PYTHONPATH=ROOT)
        out = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, check=True)
        assert out.stdout.strip() == want


def test_paths_without_a_deterministic_variant_raise_or_warn(recorder):
    config.check_deterministic("anything")           # off: nothing happens
    with config.using(deterministic=True):
        with pytest.raises(RuntimeError, match="no deterministic variant"):
            config.check_deterministic("the SIMT kernels")
        # fp32 mode and attn_impl simt select the SIMT backward, which refuses at the call (before touching the device)
        for kw in ({"mode": "fp32"}, {"attn_impl": "simt"}):
            with config.using(**kw):
                assert config.attn_impl("bwd") == 0
                geom = ops.Geometry.get(130, [32, 64, 128, 256, 512], [1, 2, 4, 8, 16])
                dattn = torch.zeros(geom.n_alloc, 768)
                with pytest.raises(RuntimeError, match="SIMT dilated-attention backward"):
                    ops.dilated_attn_bwd(geom, None, dattn, None, None, 0)
        t = torch.zeros(4, 192)
        with pytest.raises(RuntimeError, match="SIMT cross-attention backward"):
            ops.cross_attn_bwd(t, t, t, t, t, None, 12, impl=0)
    assert recorder.calls == []
    # torch's flag with warn_only: a warning instead
    torch.use_deterministic_algorithms(True, warn_only=True)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        config.check_deterministic("the SIMT kernels")
    assert any("no deterministic variant" in str(x.message) for x in w)
    # ...but the project's own switch always raises
    with config.using(deterministic=True):
        with pytest.raises(RuntimeError):
            config.check_deterministic("the SIMT kernels")


class _Recorder:
    """Stands in for the shared library: records which entry points ops calls."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def fn(*args):
            self.calls.append(name)
            return 64 if name.endswith("workspace_floats") else 0
        return fn


@pytest.fixture
def recorder(monkeypatch):
    rec = _Recorder()
    monkeypatch.setattr(_lib, "load", lambda: rec)
    monkeypatch.setattr(ops, "_p", lambda t: None)
    monkeypatch.setattr(ops, "_ptr", lambda t: None)
    monkeypatch.setattr(ops, "_rows_ok", lambda t: None)
    monkeypatch.setattr(ops, "_stream", lambda: None)
    return rec


def test_ops_select_workspace_entry_points_only_in_deterministic_mode(recorder):
    x = torch.zeros(2048, 768)
    g = torch.zeros(768)
    t = torch.zeros(100, 192)
    kv = torch.zeros(66, 192)
    for det in (False, True):
        recorder.calls.clear()
        with config.using(deterministic=det):
            ops.layernorm_bwd(x, x, g, g, g, torch.float32, want_wgrad=True)
            ops.gated_residual_bwd(x, x, x, g, want_dysum=True)
            ops.cross_attn_bwd(t, kv, kv, t, t, None, 12, impl=1)
        ws = [c for c in recorder.calls if c.endswith("_ws")]
        if det:
            assert ws == ["mt_layernorm_bwd_ws", "mt_gated_residual_bwd_ws", "mt_cross_attn_bwd_ws"], recorder.calls
        else:
            assert ws == [] and "mt_layernorm_bwd" in recorder.calls and "mt_cross_attn_bwd" in recorder.calls


def test_captured_step_signature_follows_the_switch():
    stub = type("Stub", (), {})()
    stub.model = torch.nn.Linear(2, 2)
    stub._frozen_signature = lambda: train_step.GraphedStep._frozen_signature(stub)
    a = train_step.GraphedStep._capture_signature(stub)
    with config.using(deterministic=not config.deterministic()):
        b = train_step.GraphedStep._capture_signature(stub)
    assert a != b and a[1] == b[1]


def test_header_declares_the_deterministic_entry_points():
    for name in ("mt_layernorm_bwd_ws", "mt_gated_residual_bwd_ws", "mt_colsum_ws", "mt_colreduce_workspace_floats",
                 "mt_cross_attn_bwd_ws", "mt_cross_attn_bwd_workspace_floats"):
        assert name in _lib.SIGNATURES
    text = open(os.path.join(ROOT, "include", "modaltune_b200.h")).read()
    assert "#define MT_DILATED_BWD_DETERMINISTIC 4" in text
    assert config.DETERMINISTIC_BWD_IMPL == 4
    if os.path.exists(_lib.LIB_PATH):
        lib = ctypes.CDLL(_lib.LIB_PATH)
        for name in _lib.SIGNATURES:
            assert hasattr(lib, name), name
        # workspace sizes are pure host arithmetic: 2 x 296 block partials per column
        fn = lib.mt_colreduce_workspace_floats
        fn.restype, fn.argtypes = ctypes.c_int64, [ctypes.c_int64]
        assert fn(768) == 2 * 296 * 768
