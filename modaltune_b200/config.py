"""Run-time switches of the compute path.

``mode``
    ``"bf16"`` -- fp32 residual stream, LayerNorm / softmax / GELU statistics in fp32, bf16 GEMM and attention operands
    with fp32 accumulation (the same structure the reference has under ``autocast``, SURVEY.md appendix A.6);
    ``"fp32"`` -- everything in fp32 (cuBLAS fp32 GEMMs without TF32, fp32 SIMT attention); the 1e-4 parity mode.
``attn_impl``
    ``"auto"`` -- tcgen05/TMA dilated-attention kernels in bf16 mode, SIMT kernels in fp32 mode;
    ``"simt"`` -- force the SIMT kernels (any mode);  ``"sm100"`` -- force the tcgen05 kernels (bf16 only).
``deterministic``
    bitwise-reproducible backward: every gradient reduction of the project's kernels runs in a fixed order, so the same
    seeded step gives the same loss, logits, gradients and optimizer updates in every run.  On with
    ``MODALTUNE_B200_DETERMINISTIC=1``, ``using(deterministic=True)`` or ``torch.use_deterministic_algorithms(True)``.
"""
from __future__ import annotations

import contextlib
import os
import warnings

import torch

_state = {
    "mode": os.environ.get("MODALTUNE_B200_MODE", "bf16"),
    "attn_impl": os.environ.get("MODALTUNE_B200_ATTN", "auto"),
    # the three task passes of a step on separate CUDA streams (parallel branches of the captured graph): ~8 % faster
    # at 10k tiles; MODALTUNE_B200_PASS_STREAMS=0 runs them back to back on one stream
    "pass_streams": os.environ.get("MODALTUNE_B200_PASS_STREAMS", "1") != "0",
    # frozen linear layers of the encoder in bf16 mode: "sm100" = the hand-written tcgen05 GEMM with fused epilogues
    # (mt_linear_sm100), "cublas" = library GEMMs + separate element-wise kernels (the round-1 path, kept for comparison)
    "gemm": os.environ.get("MODALTUNE_B200_GEMM", "sm100"),
    # backward of GELU + ffn_layernorm inside the epilogue of fc2's dX GEMM (MT_EPI_GELU_LN_BWD); "0" = the separate
    # GELU'-LN' kernel between two plain dX GEMMs (the path before, kept for comparison)
    "ffn_bwd_fused": os.environ.get("MODALTUNE_B200_FFN_BWD_FUSED", "1") != "0",
    # one normalisation pass + one GEMM for the k | v projections of the three extractors of the last interaction block
    # (ops.SharedKVProjectFn); "0" = every extractor normalises and projects the slide tokens itself
    "shared_extractor_kv": os.environ.get("MODALTUNE_B200_SHARED_KV", "1") != "0",
    # A / B switches of round-2 host-side restructurings (all default on; "0" = the path before)
    "injector_fused": os.environ.get("MODALTUNE_B200_INJECTOR_FUSED", "1") != "0",     # ops.InjectorFn
    "split_param_grads": os.environ.get("MODALTUNE_B200_SPLIT_GRADS", "1") != "0",     # per-pass leaf aliases
    "cross_tc": os.environ.get("MODALTUNE_B200_CROSS_TC", "1") != "0",                 # TF32 tensor-core cross-attention
    "deterministic": os.environ.get("MODALTUNE_B200_DETERMINISTIC", "0") not in ("", "0"),
}


def flag(name: str) -> bool:
    return bool(_state[name])


def shared_extractor_kv() -> bool:
    return _state["shared_extractor_kv"]


def set_shared_extractor_kv(on: bool) -> None:
    _state["shared_extractor_kv"] = bool(on)


def ffn_bwd_fused() -> bool:
    return _state["ffn_bwd_fused"]


def set_ffn_bwd_fused(on: bool) -> None:
    _state["ffn_bwd_fused"] = bool(on)


def gemm_impl() -> str:
    """Which GEMM runs the frozen encoder linears in bf16 mode (fp32 mode always uses exact fp32 cuBLAS GEMMs)."""
    return _state["gemm"] if _state["mode"] == "bf16" else "cublas"


def set_gemm_impl(impl: str) -> None:
    assert impl in ("sm100", "cublas")
    _state["gemm"] = impl


def pass_streams() -> bool:
    """Run the independent task passes of ``forward_tasks`` on separate CUDA streams."""
    return _state["pass_streams"]


def set_pass_streams(on: bool) -> None:
    _state["pass_streams"] = bool(on)


def set_mode(mode: str) -> None:
    assert mode in ("bf16", "fp32")
    _state["mode"] = mode


def set_attn_impl(impl: str) -> None:
    assert impl in ("auto", "simt", "sm100")
    _state["attn_impl"] = impl


def mode() -> str:
    return _state["mode"]


def compute_dtype() -> torch.dtype:
    return torch.bfloat16 if _state["mode"] == "bf16" else torch.float32


# what "auto" resolves to in bf16 mode, per direction: the ``impl`` selector of mt_dilated_attn_{fwd,bwd}
# (0 = SIMT fp32-math kernels, 1 = tcgen05 / TMA / TMEM kernels with one CTA per work item, 2 (backward only) = the same
# pipeline in persistent CTAs that pull items from a device counter, 3 (forward only) = 48-key score tiles: 120 TMEM
# columns and 52 KB of shared memory per CTA, FOUR CTAs per SM).  Measured on B200 at 10k / 32k tokens: the persistent
# backward is 7 - 9 % faster than the one-shot one (it runs ONE CTA per SM, so every item hand-over it overlaps is SM
# time won back); a persistent forward was 4 % SLOWER than the one-shot forward (two CTAs per SM already hide each
# other's prologue and epilogue) and has been removed; the 48-key forward is 13 % FASTER than impl 1 (0.173 against 0.197 ms at 10k tokens, 0.830
# against 0.937 ms at 32k): sixteen softmax warps per SM keep the MUFU pipe busier than eight.
AUTO_IMPL = {"fwd": 3, "bwd": 2}


# the deterministic backward of the dilated attention (mt_dilated_attn_bwd impl 4, include/modaltune_b200.h)
DETERMINISTIC_BWD_IMPL = 4


def deterministic() -> bool:
    """Is deterministic mode on: the switch (``MODALTUNE_B200_DETERMINISTIC=1`` / ``set_deterministic``) or torch's
    ``torch.use_deterministic_algorithms(True)``."""
    return _state["deterministic"] or torch.are_deterministic_algorithms_enabled()


def set_deterministic(on: bool) -> None:
    _state["deterministic"] = bool(on)


def check_deterministic(what: str) -> None:
    """``what`` has no deterministic variant: in deterministic mode raise, as torch does for its own ops (or warn when
    torch's flag is set with ``warn_only=True``)."""
    if not deterministic():
        return
    msg = (f"{what} adds gradients in arbitrary order and has no deterministic variant; deterministic mode needs bf16 "
           "mode with the tcgen05 attention kernels (attn_impl auto / sm100) and the tensor-core cross-attention")
    if not _state["deterministic"] and torch.is_deterministic_algorithms_warn_only_enabled():
        warnings.warn(msg)
        return
    raise RuntimeError(msg)


def attn_impl(direction: str = "fwd") -> int:
    """The ``impl`` argument of mt_dilated_attn_{fwd,bwd}: 0 = SIMT, 1 / 2 = tcgen05 (forward: O accumulated in TMEM
    with a lazily raised row maximum; backward: transposed formulation, per-query statistics folded into the MMAs, TMA
    reduce-adds for dQ / dK / dV), 2 = persistent CTAs.  In deterministic mode ``ops.dilated_attn_bwd`` runs the
    tcgen05 backward as impl 4 (``DETERMINISTIC_BWD_IMPL``)."""
    impl = _state["attn_impl"]
    if impl == "simt" or _state["mode"] == "fp32":
        if impl == "sm100":
            raise RuntimeError("the tcgen05 dilated-attention kernels compute in bf16; fp32 mode needs attn_impl simt/auto")
        return 0
    return AUTO_IMPL[direction]


@contextlib.contextmanager
def using(mode: str | None = None, attn_impl: str | None = None, gemm: str | None = None,
          deterministic: bool | None = None):
    old = dict(_state)
    try:
        if mode is not None:
            set_mode(mode)
        if attn_impl is not None:
            set_attn_impl(attn_impl)
        if gemm is not None:
            set_gemm_impl(gemm)
        if deterministic is not None:
            set_deterministic(deterministic)
        yield
    finally:
        _state.update(old)
