"""Fused Adam with torch.optim.Adam's interface and state_dict layout.

The reference builds its optimizer as `optim.Adam(model.parameters(), lr=learning_rate)` (train.py:163,
train_iterable.py:180) and only ever calls zero_grad(), step(), state_dict() and param_groups[0]['lr']
(train.py:184,193,196,211). `Adam` below keeps exactly that surface; step() is one rvae_adam_step launch over the
model's flat parameter buffer (28 B/param of HBM traffic) that also refreshes the bf16 shadow weights.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import _lib, engine, ops


class Adam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0, amsgrad=False):
        if amsgrad:
            raise NotImplementedError("amsgrad is not implemented by the fused kernel (the reference never uses it)")
        if not 0.0 <= lr:
            raise ValueError(f"Invalid learning rate: {lr}")
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False, maximize=False,
                        foreach=None, capturable=False, differentiable=False, fused=None)
        super().__init__(params, defaults)
        self._flat: Optional[engine.FlatState] = None
        self._loose: Dict[int, dict] = {}   # state of parameters that are not part of a VAE flat buffer

    # ------------------------------------------------------------------ flat binding
    def bind_flat(self, flat: engine.FlatState) -> None:
        """Expose the flat Adam moments as per-parameter state entries (views), torch.optim.Adam format."""
        if self._flat is flat:
            return
        self._flat = flat
        for group in self.param_groups:
            for p in group["params"]:
                tag = engine.flat_of(p)
                if tag is None or tag[0] is not flat:
                    continue
                name = tag[1]
                self.state[p] = {"step": flat.step, "exp_avg": flat.view(flat.exp_avg, name),
                                 "exp_avg_sq": flat.view(flat.exp_avg_sq, name)}

    def _find_flat(self) -> Optional[engine.FlatState]:
        flat = None
        for group in self.param_groups:
            for p in group["params"]:
                tag = engine.flat_of(p)
                if tag is None:
                    return None
                f, name = tag
                off, _ = f.offsets[name]
                if p.data_ptr() != f.params.data_ptr() + 4 * off:
                    return None  # the parameter was moved after flattening
                if flat is None:
                    flat = f
                elif flat is not f:
                    return None
        return flat

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        params = [p for g in self.param_groups for p in g["params"]]
        if any(not p.is_cuda for p in params):
            raise _lib.RvaeError("fused Adam: parameters must live on the GPU (no CPU fallback)")
        g = self.param_groups[0]
        b1, b2 = g["betas"]
        flat = self._find_flat() if len(self.param_groups) == 1 else None
        if flat is not None and len(params) == len(flat.offsets):
            self.bind_flat(flat)
            if all(p.grad is None for p in params):
                return loss
            g0 = flat.grads.data_ptr()
            for p in params:
                _, name = engine.flat_of(p)
                off, _ = flat.offsets[name]
                view = flat.view(flat.grads, name)
                if p.grad is None:
                    view.zero_()
                elif p.grad.data_ptr() != g0 + 4 * off:
                    view.copy_(p.grad)          # gradient produced elsewhere (e.g. accumulated): stage it
            ops.adam_step(flat.params, flat.grads, flat.exp_avg, flat.exp_avg_sq, flat.step, g["lr"], b1, b2,
                          g["eps"], g["weight_decay"], 1.0, flat.shadow_hi, flat.shadow_lo)
            return loss
        # generic tensors: same kernel, one launch per parameter
        for group in self.param_groups:
            b1, b2 = group["betas"]
            for p in group["params"]:
                if p.grad is None:
                    continue
                st = self.state[p]
                if len(st) == 0:
                    st["step"] = torch.zeros((), dtype=torch.float32, device=p.device)
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                if p.dtype != torch.float32:
                    raise _lib.RvaeError("fused Adam: parameters must be float32")
                # a VAE parameter of a padded model is a strided view of its block: update a contiguous copy
                pc = p.data if p.is_contiguous() else p.data.contiguous()
                ops.adam_step(pc.view(-1), p.grad.contiguous().view(-1), st["exp_avg"].view(-1),
                              st["exp_avg_sq"].view(-1), st["step"], group["lr"], b1, b2, group["eps"],
                              group["weight_decay"])
                if pc is not p.data:
                    p.data.copy_(pc)
                tag = engine.flat_of(p)
                if tag is not None:
                    tag[0].shadow_version = -1  # shadows are stale; refreshed at the next forward
        return loss

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        flat, self._flat = self._flat or self._find_flat(), None
        if flat is None:
            return
        step = None
        for group in self.param_groups:
            for p in group["params"]:
                tag = engine.flat_of(p)
                st = self.state.get(p)
                if tag is None or not st:
                    continue
                flat.view(flat.exp_avg, tag[1]).copy_(st["exp_avg"])
                flat.view(flat.exp_avg_sq, tag[1]).copy_(st["exp_avg_sq"])
                step = float(st["step"])
        if step is not None:
            flat.step.fill_(step)
        self.bind_flat(flat)
