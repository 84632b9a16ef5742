"""Run-time switches of the engine (process-wide)."""
from __future__ import annotations

import os

_state = {
    # "bf16": fused tcgen05 kernel (throughput mode, <=1e-2 parity); "fp32": SIMT parity mode (<=1e-4);
    # "bf16x3": error-compensated bf16 on the tensor cores (<=1e-4 parity at a few hundred TFLOP/s); Trainer steps run
    # its tensor-core backward too, autograd calls that need gradients run the fp32 kernels (ops.mlp_apply)
    "precision": os.environ.get("NERF_B200_PRECISION", "bf16"),
    # "reference": draw torch.rand(B,N) from the CPU global generator exactly like
    # utils/rendering.py:28 (bit-identical ts);  "philox": counter-based generator on the device.
    "sampler": os.environ.get("NERF_B200_SAMPLER", "reference"),
    "seed": int(os.environ.get("NERF_B200_SEED", "1")),
    "philox_offset": 0,
    # fp32 mode keeps ~10 KB/sample for backward; chunk the MLP to bound workspace
    # render loops: False = sampler, fused posenc+MLP and compositing as separate kernels (measured 2 % FASTER on
    # B200: the MLP kernel is bound by its epilogue warps / the power cap, and the fused kernel adds the sampler
    # and compositing work to exactly those warps); True = one kernel per chunk (no per-sample HBM traffic)
    "fused_render": os.environ.get("NERF_B200_FUSED_RENDER", "0") == "1",
    # RayGenerator.select: "reference" = CPU randperm over the whole ray table like utils/dataload.py:151
    # (328 ms per step at 4 M rays); "device" = Philox indices with replacement + gather on the GPU,
    # rays returned on the device, only the ids (8 B/ray) come back to the host for train.py:49
    "select": os.environ.get("NERF_B200_SELECT", "reference"),
    "max_samples_per_call": int(os.environ.get("NERF_B200_MAX_SAMPLES", str(1 << 22))),
}


def set_precision(p: str):
    if p not in ("bf16", "fp32", "bf16x3", "bf16_layerwise"):
        raise ValueError("precision must be 'bf16', 'fp32', 'bf16x3' or 'bf16_layerwise'")
    _state["precision"] = p


def get_precision() -> str:
    return _state["precision"]


def set_sampler(mode: str, seed: int | None = None):
    if mode not in ("reference", "philox"):
        raise ValueError("sampler must be 'reference' or 'philox'")
    _state["sampler"] = mode
    if seed is not None:
        _state["seed"] = int(seed)
        _state["philox_offset"] = 0


def get_sampler() -> str:
    return _state["sampler"]


def next_philox(n_samples: int):
    """Reserve a counter range for n_samples draws; returns (seed, offset)."""
    off = _state["philox_offset"]
    _state["philox_offset"] = off + (n_samples + 3) // 4
    return _state["seed"], off


def set_fused_render(on: bool):
    _state["fused_render"] = bool(on)


def get_fused_render() -> bool:
    return _state["fused_render"]


def set_select(mode: str):
    if mode not in ("reference", "device"):
        raise ValueError("select must be 'reference' or 'device'")
    _state["select"] = mode


def get_select() -> str:
    return _state["select"]
