"""Exponential moving average (EMA) of the VAE's weights, kept on the GPU.

`ExponentialMovingAverage(model, decay)` is torch.optim.swa_utils.AveragedModel(model,
multi_avg_fn=get_ema_multi_avg_fn(decay)) with `update_parameters(model)` after every optimizer step:

    n_averaged == 0:  e = p              otherwise:  e = torch.lerp(e, p, 1 - decay)
    n_averaged += 1

Pass it to FusedTrainStep / DataParallelTrainStep (`ema=`) and the fused Adam launches of every step update it from
the parameters they have just computed (rvae_plan_set_ema): no extra launch, no host round trip, and captured CUDA
graphs keep updating it. On the unfused path call `ema.update()` after `optimizer.step()` (rvae_ema_update).

`ema.module` is a VAE of the model's dims and precision whose flat fp32 parameter buffer IS the average, so it
encodes, decodes, evaluates and reconstructs with the averaged weights - the ones usually listened to and shipped.
"""
from __future__ import annotations

import math
from typing import Dict

import torch

from . import _lib, ops


def check_ema_decay(value) -> float:
    """An EMA decay: a number in [0, 1], as torch's get_ema_multi_avg_fn accepts. Raises ValueError for anything else."""
    if isinstance(value, bool) or not isinstance(value, (int, float)):
        raise ValueError(f"ema decay must be a number in [0, 1], got {value!r}")
    v = float(value)
    if math.isnan(v) or not 0.0 <= v <= 1.0:
        raise ValueError(f"ema decay must be in [0, 1], got {value!r}")
    return v


class ExponentialMovingAverage:
    """The EMA of `model`'s weights (a CUDA `VAE`), starting from a copy of them.

    decay (settable): weight 1 - decay of each new step. A step reads it from its device record when its kernels
    run, so a change reaches captured graphs without a new capture. n_averaged: the device int64 update count.
    module: the averaged VAE; its bf16 shadow weights are refreshed on its next use after any update. Do not move
    it to another device or precision: the buffer the kernels write is its flat parameter buffer."""

    def __init__(self, model, decay: float = 0.999):
        self._decay = check_ema_decay(decay)
        from .model import VAE
        if not model.fc1.weight.is_cuda:
            raise _lib.RvaeError("ExponentialMovingAverage needs a CUDA model - there is no CPU fallback")
        dev = model.fc1.weight.device
        self.module = VAE(model.segment_length, model.n_units, model.latent_dim, precision=model.precision).to(dev)
        self.module.eps_source, self.module.eps_seed = model.eps_source, model.eps_seed
        with torch.no_grad():
            src = model._ensure_flat()
            self.buffer().copy_(src.params)
        self.n_averaged = torch.zeros((), dtype=torch.int64, device=dev)
        self._decay_dev = torch.full((), self._decay, dtype=torch.float64, device=dev)
        self.model = model

    @property
    def decay(self) -> float:
        return self._decay

    @decay.setter
    def decay(self, value):
        self._decay = check_ema_decay(value)
        self._decay_dev.fill_(self._decay)

    def buffer(self) -> torch.Tensor:
        """The average: the fp32 flat parameter buffer of `module` (padded layout of engine.FlatState)."""
        return self.module._ensure_flat().params

    def target(self) -> torch.Tensor:
        """The same buffer without refreshing module's shadows (what a training step hands to its kernels)."""
        flat = self.module._flat
        return flat.params if flat is not None else self.buffer()

    def mark_updated(self) -> None:
        """Updates were enqueued since the last use of `module`: refresh its bf16 shadows on the next one (kernel
        writes do not bump the parameters' version counters)."""
        flat = self.module._flat
        if flat is not None:
            flat.shadow_version = -1

    def update(self) -> None:
        """One EMA update from the model's current parameters (AveragedModel.update_parameters), one launch."""
        flat = self.model._ensure_flat()
        e = self.target()
        if flat.device != e.device:
            raise _lib.RvaeError("the EMA and the model are on different devices")
        ops.ema_update(e, flat.params, self._decay_dev, self.n_averaged)
        self.mark_updated()

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """The averaged weights under the reference VAE's keys (fc1.weight, ..., unpadded contiguous copies)."""
        return {k: v.detach().clone() for k, v in self.module.state_dict().items()}

    def load_state_dict(self, state_dict, n_averaged=None) -> None:
        """Restore the average (reference keys) and, when given, n_averaged (an int or a 0-dim tensor)."""
        self.module.load_state_dict(state_dict)
        if n_averaged is not None:
            self.n_averaged.fill_(int(n_averaged))
