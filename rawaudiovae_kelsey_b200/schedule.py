"""Learning-rate and KL-weight schedules of the fused training steps.

The reference trains at a fixed learning rate (torch.optim.Adam, train.py:163,193) and a fixed KL weight
(rawvae/model.py:45). A `Schedule` adds a learning-rate warm-up and a linear or cosine decay, and a linear or
cyclical ramp of the KL weight beta (Bowman et al. 2016; Fu et al. 2019). FusedTrainStep and DataParallelTrainStep
keep the hyper-parameters in a small device record (rvae_hparams, include/rvae_b200.h) that the kernels read when
they run, so captured CUDA graphs follow the schedule step by step.

`lr_at` and `beta_at` are the host mirror of the device function: the same fp64 operations in the same order (python
floats do not contract a * b + c), so they return the doubles the kernels compute, bit for bit.
"""
from __future__ import annotations

import ctypes as C
import math
import struct
from dataclasses import dataclass

import torch

from . import _lib

LR_SCHEDULES = {"constant": 0, "linear": 1, "cosine": 2}
KL_ANNEALS = {"constant": 0, "linear": 1, "cyclical": 2}

# (-1)^n / (2n)!: the Taylor series of cos to x^22, the polynomial the kernels evaluate (csrc/elementwise.cu)
_COS_TAYLOR = tuple((-1) ** n / math.factorial(2 * n) for n in range(12))


def _cos_pi_unit(u: float) -> float:
    """cos(pi u) for u in [0, 1], operation by operation as cos_pi_unit in csrc/elementwise.cu."""
    flip = u > 0.5
    if flip:
        u = 1.0 - u
    x = math.pi * u
    x2 = x * x
    r = _COS_TAYLOR[11]
    for c in reversed(_COS_TAYLOR[:11]):
        r = r * x2 + c
    return -r if flip else r


def _integral(name, v, lo):
    if isinstance(v, bool) or not isinstance(v, (int, float)) or v != int(v):
        raise ValueError(f"{name} must be an integer, got {v!r}")
    if int(v) < lo:
        raise ValueError(f"{name} must be >= {lo}, got {v!r}")
    return int(v)


def _finite(name, v):
    v = float(v)
    if not math.isfinite(v):
        raise ValueError(f"{name} must be finite, got {v!r}")
    return v


@dataclass(frozen=True)
class Schedule:
    """lr(k) and beta(k) as closed-form functions of the step index k (the optimizer's step counter when the step
    starts; Adam's bias correction keeps t = k + 1). T = total_steps, W = warmup_steps.

    Learning rate: lr * (k + 1) / W for k < W; after that, with D = max(T - W, 1) and u = min(k - W, D) / D,
    `constant` lr, `linear` lr_min + (lr - lr_min) * (1 - u), `cosine` lr_min + (lr - lr_min) * 0.5 * (1 + cos(pi u)).
    Steps past T hold the final value.

    KL weight: `constant` kl_beta, `linear` b0 + (kl_beta - b0) * min(1, k / kl_anneal_steps), `cyclical` with
    C = ceil(T / kl_cycles) and tau = (k mod C) / C: b0 + (kl_beta - b0) * min(1, tau / kl_cycle_ratio), where
    b0 = kl_beta_start.

    The peak values lr and kl_beta are not part of the schedule: the training step takes them from
    optimizer.param_groups[0] and its kl_beta. The default schedule trains at those values, as the reference does."""
    lr_schedule: str = "constant"
    warmup_steps: int = 0
    total_steps: int = 0
    lr_min: float = 0.0
    kl_anneal: str = "constant"
    kl_beta_start: float = 0.0
    kl_anneal_steps: int = 1
    kl_cycles: int = 1
    kl_cycle_ratio: float = 0.5

    def __post_init__(self):
        if self.lr_schedule not in LR_SCHEDULES:
            raise ValueError(f"lr_schedule must be one of {sorted(LR_SCHEDULES)}, got {self.lr_schedule!r}")
        if self.kl_anneal not in KL_ANNEALS:
            raise ValueError(f"kl_anneal must be one of {sorted(KL_ANNEALS)}, got {self.kl_anneal!r}")
        decays = self.lr_schedule != "constant" or self.kl_anneal == "cyclical"
        fix = lambda name, v: object.__setattr__(self, name, v)   # noqa: E731 (frozen dataclass)
        fix("warmup_steps", _integral("warmup_steps", self.warmup_steps, 0))
        fix("total_steps", _integral("total_steps", self.total_steps, 1 if decays else -2 ** 63))
        fix("kl_anneal_steps", _integral("kl_anneal_steps", self.kl_anneal_steps,
                                         1 if self.kl_anneal == "linear" else -2 ** 63))
        fix("kl_cycles", _integral("kl_cycles", self.kl_cycles, 1 if self.kl_anneal == "cyclical" else -2 ** 63))
        fix("lr_min", _finite("lr_min", self.lr_min))
        fix("kl_beta_start", _finite("kl_beta_start", self.kl_beta_start))
        fix("kl_cycle_ratio", _finite("kl_cycle_ratio", self.kl_cycle_ratio))
        if not 0.0 < self.kl_cycle_ratio <= 1.0:
            raise ValueError(f"kl_cycle_ratio must be in (0, 1], got {self.kl_cycle_ratio!r}")

    def lr_at(self, k: int, lr: float) -> float:
        """Learning rate at step index k for the peak learning rate lr (fp64, as Adam receives it)."""
        k, lr, W = int(k), float(lr), self.warmup_steps
        if k < W:
            return lr * (k + 1) / W
        if self.lr_schedule == "constant":
            return lr
        D = max(self.total_steps - W, 1)
        u = min(k - W, D) / D
        span = lr - self.lr_min
        if self.lr_schedule == "linear":
            return self.lr_min + span * (1.0 - u)
        return self.lr_min + span * 0.5 * (1.0 + _cos_pi_unit(u))

    def beta_at(self, k: int, kl_beta: float) -> float:
        """KL weight at step index k for the target kl_beta, in fp64 (the kernels round it to fp32)."""
        k, kl_beta = int(k), float(kl_beta)
        if self.kl_anneal == "constant":
            return kl_beta
        if self.kl_anneal == "linear":
            f = min(1.0, k / self.kl_anneal_steps)
        else:
            c = -(-self.total_steps // self.kl_cycles)
            f = min(1.0, (k % c) / c / self.kl_cycle_ratio)
        b0 = self.kl_beta_start
        return b0 + (kl_beta - b0) * f

    def record(self, lr, betas, eps, weight_decay, kl_beta) -> _lib.Hparams:
        """The rvae_hparams record of this schedule with these peak values. Raises ValueError for a non-finite value."""
        b1, b2 = betas
        vals = {n: _finite(n, v) for n, v in (("lr", lr), ("beta1", b1), ("beta2", b2), ("eps", eps),
                                              ("weight_decay", weight_decay), ("kl_beta", kl_beta))}
        return _lib.Hparams(lr_min=self.lr_min, kl_beta_start=self.kl_beta_start, kl_cycle_ratio=self.kl_cycle_ratio,
                            total_steps=self.total_steps, warmup_steps=self.warmup_steps,
                            kl_anneal_steps=self.kl_anneal_steps, kl_cycles=self.kl_cycles,
                            lr_schedule=LR_SCHEDULES[self.lr_schedule], kl_anneal=KL_ANNEALS[self.kl_anneal], **vals)


class DeviceRecord:
    """The device copy of a training step's rvae_hparams record, followed by the gradient-clipping threshold and the
    EMA decay (two doubles; rvae_plan_set_grad_clip, rvae_plan_set_ema). `update` rewrites all three - with one copy
    from pinned memory, ordered on the current stream, without a device synchronisation - only when the schedule, a
    peak value, the threshold or the decay differs from what the record holds. The record keeps its address, so a
    captured graph reads the new values."""

    def __init__(self, device):
        self.tensor = torch.zeros(C.sizeof(_lib.Hparams) + 16, dtype=torch.uint8, device=device)
        self._key = None

    @property
    def max_norm_ptr(self) -> int:
        """Device address of the clipping threshold."""
        return self.tensor.data_ptr() + C.sizeof(_lib.Hparams)

    @property
    def ema_decay_ptr(self) -> int:
        """Device address of the EMA decay."""
        return self.tensor.data_ptr() + C.sizeof(_lib.Hparams) + 8

    def update(self, schedule: Schedule, lr, betas, eps, weight_decay, kl_beta, max_grad_norm=None,
               ema_decay=None) -> torch.Tensor:
        max_norm = math.inf if max_grad_norm is None else float(max_grad_norm)
        decay = 0.0 if ema_decay is None else float(ema_decay)
        key = (schedule, float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), float(kl_beta),
               max_norm, decay)
        if key != self._key:
            rec = schedule.record(lr, betas, eps, weight_decay, kl_beta)
            _lib.check(_lib.load().rvae_hparams_check(C.byref(rec)))
            raw = bytes(rec) + struct.pack("<dd", max_norm, decay)
            host = torch.frombuffer(bytearray(raw), dtype=torch.uint8).pin_memory()
            self.tensor.copy_(host, non_blocking=True)
            self._key = key
        return self.tensor
