"""Drop-in for the reference's rawvae/model.py: `VAE` and `loss_function` with the same names, signatures and
tensor semantics, computed by the sm_100a kernels behind include/rvae_b200.h.

Reference contract mirrored here (file:line in kelseyicotton/rawaudiovae_kelsey):
  VAE.__init__(segment_length, n_units, latent_dim)        rawvae/model.py:6-17   (same submodule names / init order)
  VAE.encode(x) -> (mu, logvar)                            rawvae/model.py:19-21
  VAE.reparameterize(mu, logvar) -> z                      rawvae/model.py:23-26
  VAE.decode(z) -> x_hat                                   rawvae/model.py:28-30
  VAE.forward(x) -> (x_hat, mu, logvar), x.view(-1, S)     rawvae/model.py:32-35
  loss_function(recon_x, x, mu, logvar, kl_beta, S)        rawvae/model.py:38-46

CUDA tensors only: CPU inputs raise (the north star forbids a CPU fallback). Parameters stay fp32 nn.Parameters
named fc1/fc21/fc22/fc3/fc4 so checkpoints load both ways; they are views into one flat buffer (engine.FlatState)
so the fused Adam kernel and the gradient all-reduce see contiguous memory.
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import _lib, engine, ops
from .schedule import DeviceRecord, Schedule

_PRIVATE = ("_flat", "_plans", "_eps_counter")


_SPAN_ON = os.environ.get("RVAE_SPAN", "1") not in ("0", "")


class FrameBatch:
    """A batch described by frame indices into a device-resident wav buffer (produced by dataset.GpuFrameLoader).
    Passing it to VAE.forward / FusedTrainStep fuses framing into the batch load: frames are gathered straight into
    the bf16 operand buffer of fc1 and never materialised as an fp32 [B, S] tensor."""

    def __init__(self, audio: torch.Tensor, n_frames: int, hop: int, segment_length: int,
                 frame_idx: Optional[torch.Tensor] = None, first_frame: int = 0,
                 global_row0: Optional[int] = None, global_batch: Optional[int] = None, run: bool = False):
        self.audio, self.n_frames, self.hop, self.segment_length = audio, int(n_frames), int(hop), int(segment_length)
        self.frame_idx, self.first_frame = frame_idx, int(first_frame)
        # run=True with a frame_idx tensor: the frames are the RUN frame_idx[0], frame_idx[0] + 1, ... (the first
        # frame lives in device memory so that a captured CUDA graph follows a stream); frame_idx=None is always a run
        self.run = bool(run) or frame_idx is None
        # data parallelism: this batch is rows [global_row0, global_row0 + n_frames) of a global batch of
        # `global_batch` frames (set by the sharding loaders; None = not sharded / equal shards assumed)
        self.global_row0, self.global_batch = global_row0, global_batch

    @property
    def shape(self):
        return (self.n_frames, self.segment_length)

    @property
    def span(self) -> bool:
        """A run of consecutive frames whose hop gives 16-byte row pitches is read IN PLACE: its contiguous sample
        span is converted to bf16 once and fc1 / the MSE / the fc1 weight gradient read frame i at row pitch hop
        through overlapping-row TMA tensor maps (rvae_plan_load_span) - same results as the gather, bit for bit.
        RVAE_SPAN=0 turns it off (A/B measurements)."""
        return (self.run and _SPAN_ON and self.hop % 8 == 0 and 0 < self.hop <= self.segment_length
                and self.segment_length % 8 == 0)

    def __len__(self):
        return self.n_frames

    def to(self, *args, **kwargs):  # `data.to(device)` in the training loops is a no-op for a device batch
        return self

    def materialize(self) -> torch.Tensor:
        """fp32 [B, S] frames (what the reference's DataLoader would have produced)."""
        idx, first = self.frame_idx, self.first_frame
        if idx is not None and self.run:
            idx, first = None, int(idx[0].item())
        f32, _, _ = ops.frame_gather(self.audio, self.n_frames, self.hop, self.segment_length,
                                     frame_idx=idx, first_frame=first)
        return f32

    def view(self, *shape):
        return self.materialize().view(*shape)


class VAE(nn.Module):
    __module__ = "rawvae.model"  # whole-module pickles (best_model.pt / last_model.pt) resolve like the reference's

    def __init__(self, segment_length, n_units, latent_dim, precision: str = "bf16"):
        super(VAE, self).__init__()
        self.segment_length = segment_length
        self.n_units = n_units
        self.latent_dim = latent_dim
        # same creation order as the reference => identical default init for a given torch.manual_seed
        self.fc1 = nn.Linear(segment_length, n_units)
        self.fc21 = nn.Linear(n_units, latent_dim)
        self.fc22 = nn.Linear(n_units, latent_dim)
        self.fc3 = nn.Linear(latent_dim, n_units)
        self.fc4 = nn.Linear(n_units, segment_length)
        self.precision = precision      # "bf16" (bf16 operands, fp32 accumulate) or "fp32" (split-bf16, 3 passes)
        self.eps_source = "philox"      # "philox": in-library Philox noise; "torch": torch.randn on the CUDA generator
        self.eps_seed = None            # philox seed (default: torch.initial_seed())
        self._flat: Optional[engine.FlatState] = None
        self._plans: Dict[int, engine.Plan] = {}
        self._eps_counter = 0

    # ------------------------------------------------------------------ pickling / device moves
    def __getstate__(self):
        state = self.__dict__.copy()
        for k in _PRIVATE:
            state.pop(k, None)
        return state

    def __setstate__(self, state):
        super().__setstate__(state)
        self.__dict__.setdefault("precision", "bf16")
        self.__dict__.setdefault("eps_source", "philox")
        self.__dict__.setdefault("eps_seed", None)
        self._flat, self._plans, self._eps_counter = None, {}, 0

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        self._flat, self._plans = None, {}
        p = self.fc1.weight
        if p.is_cuda:
            self._ensure_flat()
        return out

    def set_precision(self, precision: str) -> "VAE":
        if precision not in engine.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(engine.PRECISIONS)}")
        if precision != self.precision:
            self.precision = precision
            self._flat, self._plans = None, {}
        return self

    # ------------------------------------------------------------------ flat storage
    def _named(self) -> List:
        return [(n, p) for n, p in self.named_parameters()]

    def _ensure_flat(self) -> engine.FlatState:
        """Make every parameter a view of one flat fp32 buffer (idempotent) and keep the bf16 shadows fresh."""
        p0 = self.fc1.weight
        if not p0.is_cuda:
            raise _lib.RvaeError("VAE parameters are on the CPU: call model.to('cuda') - there is no CPU fallback")
        flat = getattr(self, "_flat", None)
        named = self._named()
        ok = flat is not None and flat.device == p0.device and flat.precision == self.precision
        if ok:
            base = flat.params.data_ptr()
            for n, p in named:
                off, shape, strides = flat.geometry[n]
                if (p.data_ptr() != base + 4 * off or tuple(p.shape) != shape or p.stride() != strides
                        or p.dtype != torch.float32):
                    ok = False
                    break
        if not ok:
            S, H, L = self.segment_length, self.n_units, self.latent_dim
            for n, p in named:
                if p.dtype != torch.float32:
                    raise _lib.RvaeError(f"parameter {n} is {p.dtype}; master weights must stay float32")
            flat = engine.FlatState(S, H, L, p0.device, self.precision)
            with torch.no_grad():
                for n, p in named:
                    v = flat.view(flat.params, n)
                    v.copy_(p.data)
                    p.data = v
                    p.grad = None
                    engine.register_flat(p, flat, n)
            self._flat, self._plans = flat, {}
            flat.shadow_version = -1
        version = sum(p._version for _, p in named)
        if version != flat.shadow_version:
            flat.sync_shadow()
            flat.shadow_version = version
        return flat

    def _in_place(self, fb: "FrameBatch") -> bool:
        """Does this model read the frames of `fb` in place (FrameBatch.span)? A segment_length that is not a multiple
        of 64 is padded inside the model; in fp32 mode such frames are gathered instead (rvae_plan_span_supported)."""
        return fb.span and (self.segment_length % 64 == 0 or self.precision == "bf16")

    def _plan_for(self, batch: int) -> engine.Plan:
        flat = self._ensure_flat()
        best = None
        for mb, pl in self._plans.items():
            if mb >= batch and (best is None or mb < best.max_batch):
                best = pl
        if best is None:
            self._plans = {}  # drop smaller workspaces
            best = engine.Plan(flat, batch)
            self._plans[batch] = best
        return best

    # ------------------------------------------------------------------ noise
    def _eps_args(self):
        seed = self.eps_seed if self.eps_seed is not None else torch.initial_seed()
        off = self._eps_counter
        self._eps_counter += 1
        return int(seed) & 0xFFFFFFFFFFFFFFFF, off

    def _set_eps(self, plan: engine.Plan, eps: Optional[torch.Tensor]) -> None:
        if eps is not None:
            plan.set_eps(eps)
        elif self.eps_source == "torch":
            plan.set_eps(torch.randn((plan.batch, self.latent_dim), device=self._flat.device))
        else:
            plan.gen_eps(*self._eps_args())

    # ------------------------------------------------------------------ reference API
    def _load(self, src):
        """Load a batch into a plan: a CUDA tensor (any shape with numel % S == 0), a FrameBatch, or a list of
        FrameBatch runs (a streaming batch that straddles files)."""
        if isinstance(src, FrameBatch):
            src = [src]
        if isinstance(src, (list, tuple)) and src and all(isinstance(r, FrameBatch) for r in src):
            total = sum(r.n_frames for r in src)
            plan = self._plan_for(total)
            row = 0
            for r in src:
                if r.segment_length != self.segment_length:
                    raise _lib.RvaeError("FrameBatch segment_length does not match the model")
                span = len(src) == 1 and self._in_place(r) and r.n_frames <= plan.max_batch
                if r.frame_idx is not None and r.run and not span:
                    raise _lib.RvaeError("a device-side run (FrameBatch(run=True)) needs hop % 8 == 0, hop <= S, "
                                         "S % 8 == 0, and bf16 precision when S % 64 != 0")
                plan.load_frames(r.audio, r.n_frames, r.hop, frame_idx=r.frame_idx, first_frame=r.first_frame,
                                 row_offset=row, span=span)
                row += r.n_frames
            return plan
        x = src
        if not isinstance(x, torch.Tensor):
            raise TypeError("expected a torch.Tensor, a FrameBatch or a list of FrameBatch")
        if not x.is_cuda:
            raise _lib.RvaeError("input is a CPU tensor: move it to the GPU - there is no CPU fallback")
        x = x.view(-1, self.segment_length)
        plan = self._plan_for(x.shape[0])
        plan.load_batch(x)
        return plan

    def encode(self, x):
        """(mu, logvar) = (fc21(relu(fc1 x)), fc22(relu(fc1 x))) - inference path, returns detached tensors."""
        plan = self._load(x)
        dev = self._flat.device
        mu = torch.empty((plan.batch, self.latent_dim), dtype=torch.float32, device=dev)
        lv = torch.empty_like(mu)
        plan.set_outputs(mu, lv, None)
        plan.encode()
        plan.set_outputs(None, None, None)
        return mu, lv

    def reparameterize(self, mu, logvar, eps: Optional[torch.Tensor] = None):
        """z = mu + eps * exp(0.5 * logvar). Accepts float64 inputs (tutorial.ipynb:922) - computed in fp32."""
        if not mu.is_cuda:
            raise _lib.RvaeError("reparameterize: CPU tensors are not supported (no CPU fallback)")
        dt = mu.dtype
        m32, l32 = mu.float().contiguous(), logvar.float().contiguous()
        if eps is None:
            if self.eps_source == "torch":
                eps = torch.randn_like(m32)
            else:
                seed, off = self._eps_args()
                eps = ops.randn(m32.shape, seed, off, device=m32.device)
        z = ops.reparameterize(m32, l32, eps.float().contiguous())
        return z.to(dt)

    def decode(self, z):
        """x_hat = tanh(fc4(relu(fc3 z))) - inference path, returns a detached tensor."""
        if not z.is_cuda:
            raise _lib.RvaeError("decode: CPU tensors are not supported (no CPU fallback)")
        z = z.reshape(-1, self.latent_dim).float().contiguous()
        plan = self._plan_for(z.shape[0])
        out = torch.empty((z.shape[0], self.segment_length), dtype=torch.float32, device=z.device)
        plan.decode(z, out)
        return out

    def reference_forward(self, x, eps: Optional[torch.Tensor] = None):
        """The forward pass as plain torch ops on the SAME parameters (rawvae/model.py:19-35, op for op): what a
        tracer can follow. The sm_100a kernels are reached through ctypes and are invisible to torch.jit.trace /
        torch.onnx.export, so `forward` routes here while it is being traced or exported
        (export-onnx.ipynb:361-362: torch.onnx.export(raw_model, torch.randn(1024), "rawaudiovae.onnx")) - an export
        path, not a compute fallback: ordinary calls never take it. Works on any device, any float dtype."""
        x = x.view(-1, self.segment_length)
        h1 = torch.relu(self.fc1(x))
        mu, logvar = self.fc21(h1), self.fc22(h1)
        std = torch.exp(0.5 * logvar)
        if eps is None:
            eps = torch.randn_like(std)
        z = mu + eps * std
        h3 = torch.relu(self.fc3(z))
        return torch.tanh(self.fc4(h3)), mu, logvar

    @staticmethod
    def _being_traced() -> bool:
        if torch.jit.is_tracing() or torch.jit.is_scripting():
            return True
        try:
            if torch.onnx.is_in_onnx_export():
                return True
        except Exception:
            pass
        is_exporting = getattr(getattr(torch, "compiler", None), "is_exporting", None)
        return bool(is_exporting and is_exporting())

    def forward(self, x, eps: Optional[torch.Tensor] = None):
        """(x_hat, mu, logvar); differentiable w.r.t. the parameters (loss.backward() works as in the reference).
        `eps` optionally injects the reparameterisation noise (parity tests); the reference draws it internally."""
        if self._being_traced():
            return self.reference_forward(x, eps)
        self._ensure_flat()
        params = [p for _, p in self._named()]
        return _VAEForward.apply(self, x, eps, *params)


class _VAEForward(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model: VAE, x, eps, *params):
        plan = model._load(x)
        model._set_eps(plan, eps)
        dev = model._flat.device
        B, S, L = plan.batch, model.segment_length, model.latent_dim
        xhat = torch.empty((B, S), dtype=torch.float32, device=dev)
        mu = torch.empty((B, L), dtype=torch.float32, device=dev)
        lv = torch.empty((B, L), dtype=torch.float32, device=dev)
        plan.set_outputs(mu, lv, xhat)
        plan.forward(0.0, fused_loss=False, want_xhat=True)
        plan.set_outputs(None, None, None)
        ctx.model, ctx.plan, ctx.token = model, plan, plan.token
        ctx.save_for_backward(xhat, lv)
        return xhat, mu, lv

    @staticmethod
    def backward(ctx, g_xhat, g_mu, g_lv):
        model, plan = ctx.model, ctx.plan
        xhat, lv = ctx.saved_tensors
        if plan.token != ctx.token:
            raise RuntimeError("the activations of this forward pass were overwritten by a later forward on the "
                               "same model; call backward() before running the model again")
        flat = model._flat
        B, L = xhat.shape[0], model.latent_dim
        z = lambda ref, shape: torch.zeros(shape, dtype=torch.float32, device=xhat.device) if ref is None \
            else ref.float().contiguous()
        g_xhat, g_mu, g_lv = z(g_xhat, xhat.shape), z(g_mu, (B, L)), z(g_lv, (B, L))
        named = model._named()
        # un-alias gradients that already live in the flat buffer (gradient accumulation / set_to_none=False)
        g0 = flat.grads.data_ptr()
        g1 = g0 + 4 * flat.total
        for _, p in named:
            if p.grad is not None and g0 <= p.grad.data_ptr() < g1:
                p.grad = p.grad.clone()
        plan.backward_external(g_xhat, xhat, g_mu, g_lv, lv)
        grads = tuple(flat.view(flat.grads, n) for n, _ in named)
        return (None, None, None) + grads


class _LossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, recon_x, x, mu, logvar, kl_beta):
        ctx.save_for_backward(recon_x, x, mu, logvar)
        ctx.kl_beta = kl_beta
        return ops.loss_fwd(recon_x, x, mu, logvar, kl_beta)

    @staticmethod
    def backward(ctx, grad_out):
        recon_x, x, mu, logvar = ctx.saved_tensors
        g = grad_out.float().contiguous() if grad_out is not None else None
        g_x, g_mu, g_lv = ops.loss_bwd(recon_x, x, mu, logvar, ctx.kl_beta, g)
        return g_x, None, g_mu, g_lv, None


# Reconstruction + KL divergence losses (mean over all elements, as the reference's mse_loss default / torch.mean)
def loss_function(recon_x, x, mu, logvar, kl_beta, segment_length):
    if isinstance(x, FrameBatch):
        x = x.materialize()
    if not recon_x.is_cuda:
        raise _lib.RvaeError("loss_function: CPU tensors are not supported (no CPU fallback)")
    x = x.view(-1, segment_length)
    c = lambda t: t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()
    return _LossFunction.apply(c(recon_x), c(x), c(mu), c(logvar), float(kl_beta))


def check_max_grad_norm(value) -> Optional[float]:
    """A training step's gradient-clipping threshold: None (no clipping) or a float > 0, +inf included (the norm is
    measured and logged, the update is unchanged). Raises ValueError for anything else."""
    if value is None:
        return None
    if isinstance(value, bool) or not isinstance(value, (int, float)):
        raise ValueError(f"max_grad_norm must be None or a number > 0, got {value!r}")
    v = float(value)
    if math.isnan(v) or v <= 0.0:
        raise ValueError(f"max_grad_norm must be > 0 (inf allowed), got {value!r}")
    return v


class _StepBase:
    """Shared machinery of FusedTrainStep / dist.DataParallelTrainStep: the device-side loss ring and the CUDA-graph
    cache. A step is enqueued by `self._enqueue(plan)` (subclass); with graph=True the enqueue is captured once per
    input signature (after `graph_warmup` eager steps) and replayed, so the host cost of a step drops from ~20
    kernel launches to one graph launch. Replays stay correct because everything that changes from step to step is
    read from device memory: frame indices from a static index buffer, the Philox offset and the loss-ring slot
    from the optimizer's step counter. The hyper-parameters too: the kernels read them from a device record
    (schedule.DeviceRecord) that each call rewrites before the step when optimizer.param_groups[0], kl_beta or
    `schedule` changed, so replays follow the schedule, a torch LR scheduler and any change made by hand.

    max_grad_norm (None = off): clip the gradient by its global L2 norm before Adam, as torch.nn.utils.clip_grad_norm_
    does, inside the step (rvae_plan_set_grad_clip). The threshold lives in the device record too, so changing
    `step.max_grad_norm` reaches graph replays; switching clipping on or off captures a new graph. The pre-clip norm
    of every step lands in a device ring of the loss ring's size; `grad_norm` is the last step's slot."""

    def __init__(self, model, optimizer, kl_beta, ring, graph, graph_warmup=1, schedule=None, max_grad_norm=None):
        self.max_grad_norm = max_grad_norm     # validated before any GPU work
        self.model, self.optimizer, self.kl_beta = model, optimizer, float(kl_beta)
        self.schedule = schedule if schedule is not None else Schedule()
        self._record = None
        self.ring_size = int(ring)
        self.ring = None
        self.norm_ring = None    # pre-clip gradient norms, slot = step counter mod ring_size (allocated when clipping)
        self.i = None            # host mirror of the device step counter (slot = i % ring_size)
        self.graph = bool(graph)
        # eager calls per input signature before its graph is captured: ONE is needed (the first call of a signature
        # builds tensor maps and tile schedules with synchronous copies, which a capture must not contain)
        self.graph_warmup = max(1, int(graph_warmup))
        self._graphs = {}        # key -> dict(graph, static buffers, plan)
        self.replayed_launches = 0   # kernels launched by graph replays (the library's launch counter only sees eager ones)
        self._seen = {}          # key -> eager calls so far
        # what each call did, so that a caller timing steady state can prove no capture / eager step fell into its
        # timed region: totals, and the number of CONSECUTIVE replayed steps up to now
        self.stats = {"eager": 0, "captures": 0, "replays": 0}
        self.steady = 0

    @property
    def max_grad_norm(self) -> Optional[float]:
        return self._max_grad_norm

    @max_grad_norm.setter
    def max_grad_norm(self, value):
        self._max_grad_norm = check_max_grad_norm(value)

    @property
    def grad_norm(self) -> Optional[torch.Tensor]:
        """The pre-clip gradient norm of the last step (0-dim device tensor, a slot of the norm ring), or None when
        clipping is off or before the first step."""
        if self.max_grad_norm is None or self.norm_ring is None or not self.i:
            return None
        return self.norm_ring[(self.i - 1) % self.ring_size]

    # -- helpers
    def _prepare(self):
        model = self.model
        flat = model._ensure_flat()
        if self.ring is None:
            self.ring = torch.zeros(self.ring_size, dtype=torch.float32, device=flat.device)
        if self.norm_ring is None and self.max_grad_norm is not None:
            self.norm_ring = torch.zeros(self.ring_size, dtype=torch.float32, device=flat.device)
        if self.i is None:
            self.i = int(flat.step.item())          # one sync, first call only (resumed optimizers start at t0 > 0)
        if hasattr(self.optimizer, "bind_flat"):
            self.optimizer.bind_flat(flat)
        return flat

    def _hparams(self, device):
        """Bring the device record up to date (outside any capture: a graph must hold its address, not a copy)."""
        if self._record is None:
            self._record = DeviceRecord(device)
        g = self.optimizer.param_groups[0]
        return self._record.update(self.schedule, g["lr"], g["betas"], g["eps"], g.get("weight_decay", 0.0),
                                   self.kl_beta, self.max_grad_norm)

    def _train_step(self, plan, zero_grads):
        """The fused step from the device record, clipping when max_grad_norm is set (a plan setting for this call)."""
        if self.max_grad_norm is None:
            plan.train_step_hp(self._record.tensor, loss_out=self.ring, ring_size=self.ring_size, zero_grads=zero_grads)
            return
        plan.set_grad_clip(self._record.max_norm_ptr, self.norm_ring, self.ring_size)
        try:
            plan.train_step_hp(self._record.tensor, loss_out=self.ring, ring_size=self.ring_size, zero_grads=zero_grads)
        finally:
            plan.set_grad_clip(None)

    def _slot(self):
        return self.ring[self.i % self.ring_size]

    def _eps(self, plan, eps):
        model = self.model
        if eps is not None:
            plan.set_eps(eps)
        elif model.eps_source == "torch":
            plan.set_eps(torch.randn((plan.batch, model.latent_dim), device=model._flat.device))
        else:
            plan.gen_eps(self._seed(), 0, add_step=True)   # offset = device step counter

    def _graph_key(self, data):
        """Input signature for graph reuse, or None when the input cannot be served by a replay."""
        if isinstance(data, FrameBatch):
            return ("frames", data.audio.data_ptr(), data.n_frames, data.hop, data.segment_length,
                    self.model._in_place(data))
        if isinstance(data, torch.Tensor) and data.is_cuda:
            return ("tensor", data.numel())
        return None

    def _load_static(self, key, data, st):
        """Refresh the static input buffers of a captured graph from this call's input."""
        if key[0] == "frames":
            if data.frame_idx is not None:
                st["idx"].copy_(data.frame_idx)
            else:
                torch.add(st["arange"], data.first_frame, out=st["idx"])
        else:
            st["x"].copy_(data.reshape(st["x"].shape))

    def _seed(self):
        model = self.model
        seed = model.eps_seed if model.eps_seed is not None else torch.initial_seed()
        return int(seed) & 0xFFFFFFFFFFFFFFFF

    def _can_prefetch(self, nxt, eps):
        model = self.model
        return (isinstance(nxt, FrameBatch) and eps is None and model.eps_source == "philox"
                and nxt.segment_length == model.segment_length)

    def _take_prefetched(self, data):
        """If `data` is the batch the previous step prefetched, make it current and return its plan."""
        pf = getattr(self, "_pf", None)
        self._pf = None
        if pf is None or pf[1] is not data:
            return None
        plan = pf[0]
        if plan.prefetched_batch() != data.n_frames:
            return None
        plan.swap_prefetched()
        return plan

    def _run(self, data, eps, next_data=None):
        """One step on `data`. `next_data` (optional FrameBatch): the batch of the NEXT call - it is gathered, and its
        noise drawn, on a background stream while this step's GEMMs run (pass the same object as `data` next time)."""
        flat = self._prepare()
        self._hparams(flat.device)
        model = self.model
        graphable = self.graph and eps is None and model.eps_source == "philox"
        plan = self._take_prefetched(data) if eps is None else None
        prefetch = plan is not None or next_data is not None
        if not prefetch:
            # ---- plain path: load inside the step (captured graph: from static index / input buffers)
            key = self._graph_key(data) if graphable else None
            if key is not None:
                key = key + self._key_extra(data) + (self.max_grad_norm is not None,)
            if key is not None and key in self._graphs:
                st = self._graphs[key]
                self._load_static(key, data, st)
                st["graph"].replay()
                self.replayed_launches += st["launches"]
                st["plan"].token += 1
                self._count("replays")
            elif key is not None and self._seen.get(key, 0) >= self.graph_warmup:
                self._capture(key, data)
                self._count("captures")
            else:
                if key is not None:
                    self._seen[key] = self._seen.get(key, 0) + 1
                plan = model._load(data)
                self._configure(plan, data)
                self._eps(plan, eps)
                self._enqueue(plan)
                self._count("eager")
        else:
            # ---- pipelined path: the current batch is already in the plan (or loaded eagerly now), the next one is
            #      prefetched by this step
            if plan is None:
                plan = model._load(data)
                self._configure(plan, data)
                self._eps(plan, eps)
            else:
                self._configure(plan, data)
            do_pf = self._can_prefetch(next_data, eps) and next_data.n_frames <= plan.max_batch
            key = None
            if graphable and do_pf and isinstance(data, FrameBatch):
                key = ("pf", plan.handle.value, next_data.audio.data_ptr(), plan.batch, next_data.n_frames,
                       next_data.hop, self._plan_cur(plan), plan.pitch, model._in_place(next_data)) \
                    + self._key_extra(data) + self._key_extra(next_data) + (self.max_grad_norm is not None,)
            if key is not None and key in self._graphs:
                st = self._graphs[key]
                self._fill_idx(st, next_data)
                st["graph"].replay()
                self.replayed_launches += st["launches"]
                self._mark_prefetched(plan, next_data)
                self._count("replays")
            elif key is not None and self._seen.get(key, 0) >= self.graph_warmup:
                self._capture_pipelined(key, plan, next_data)
                self._count("captures")
            else:
                self._count("eager")
                if key is not None:
                    self._seen[key] = self._seen.get(key, 0) + 1
                if do_pf:
                    self._prefetch(plan, data, next_data, next_data.frame_idx, next_data.first_frame)
                self._enqueue(plan)
                if do_pf:
                    self._pf = (plan, next_data)
        slot = self._slot()
        self.i += 1
        return slot

    # -- hooks of the data-parallel subclass
    def _configure(self, plan, data):
        """Per-step plan settings that depend on the batch (global batch size, first global row of the shard)."""

    def _key_extra(self, data):
        """What _configure bakes into a captured graph, as part of the graph key."""
        return ()

    def _prefetch(self, plan, data, next_data, frame_idx, first_frame):
        """Register next_data (frames + noise) as the batch the coming train step gathers in the background."""
        plan.prefetch_frames(next_data.audio, next_data.n_frames, next_data.hop, frame_idx=frame_idx,
                             first_frame=first_frame, seed=self._seed(), offset=0, add_step=True,
                             span=self.model._in_place(next_data))

    def _count(self, what):
        self.stats[what] += 1
        self.steady = self.steady + 1 if what == "replays" else 0

    def _plan_cur(self, plan):
        """Parity of the plan's current input set (captured graphs bake in its addresses): tracked on the host."""
        return plan.cur

    def _mark_prefetched(self, plan, next_data):
        # a replayed graph performed the prefetch on the device; mirror it in the plan's host-side state
        plan.note_prefetched(next_data.n_frames, next_data.hop if self.model._in_place(next_data) else 0)
        self._pf = (plan, next_data)

    def _fill_idx(self, st, nxt):
        if nxt.frame_idx is not None:
            st["idx"].copy_(nxt.frame_idx)
        else:
            torch.add(st["arange"], nxt.first_frame, out=st["idx"])

    def _capture_pipelined(self, key, plan, next_data):
        dev = self.model._flat.device
        st = {"idx": torch.empty(next_data.n_frames, dtype=torch.int64, device=dev),
              "arange": torch.arange(next_data.n_frames, dtype=torch.int64, device=dev)}
        self._fill_idx(st, next_data)
        plan.join_background()
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        l0 = ops.launch_count(dev)
        with torch.cuda.graph(g):
            self._prefetch(plan, None, next_data, st["idx"], 0)
            self._enqueue(plan)
        st["graph"], st["plan"], st["launches"] = g, plan, ops.launch_count(dev) - l0
        self._graphs[key] = st
        g.replay()   # capture does not execute: this replay performs the step of the current call
        self._pf = (plan, next_data)

    def _capture(self, key, data):
        model = self.model
        dev = model._flat.device
        st = {}
        if key[0] == "frames":
            st["idx"] = torch.empty(data.n_frames, dtype=torch.int64, device=dev)
            st["arange"] = torch.arange(data.n_frames, dtype=torch.int64, device=dev)
            static_in = FrameBatch(data.audio, data.n_frames, data.hop, data.segment_length, frame_idx=st["idx"],
                                   run=model._in_place(data))
        else:
            st["x"] = torch.empty((data.numel() // model.segment_length, model.segment_length), dtype=torch.float32,
                                  device=dev)
            static_in = st["x"]
        self._load_static(key, data, st)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        l0 = ops.launch_count(dev)
        with torch.cuda.graph(g):
            plan = model._load(static_in)
            self._configure(plan, data)
            self._eps(plan, None)
            self._enqueue(plan)
        st["graph"], st["plan"], st["launches"] = g, plan, ops.launch_count(dev) - l0
        self._graphs[key] = st
        g.replay()   # capture does not execute: this replay performs the step of the current call


class FusedTrainStep(_StepBase):
    """zero_grad + forward + loss + backward + Adam (train_iterable.py:200-210) as ONE C call: every kernel of the
    step is enqueued by rvae_plan_train_step, the loss gradients are produced by the forward epilogues, and the
    loss lands in a device-side ring so the host never has to synchronise per step.

        step = FusedTrainStep(model, optimizer, kl_beta)
        loss = step(data)            # 0-dim CUDA tensor (a slot of the ring); .item() only when you log

    keep_grads=False (default): the Adam kernel clears the flat gradient buffer after consuming it, exactly what the
    reference's optimizer.zero_grad() does at the top of the next iteration; keep_grads=True leaves the step's
    gradients in model._flat.grads for inspection (costs memsets per step). With clipping they are the raw,
    unclipped gradients: the norm torch.nn.utils.clip_grad_norm_ returns, and step.grad_norm holds, is theirs.
    graph=True: replay a captured CUDA graph of the step (see _StepBase).
    schedule (schedule.Schedule, default constant): learning rate and KL weight per step, with
    optimizer.param_groups[0]['lr'] and kl_beta as the peak values.
    max_grad_norm (None, or a float > 0, inf included): clip by the global gradient norm (see _StepBase)."""

    def __init__(self, model: VAE, optimizer, kl_beta: float, ring: int = 64, keep_grads: bool = False,
                 graph: bool = False, schedule: Optional[Schedule] = None, max_grad_norm: Optional[float] = None):
        super().__init__(model, optimizer, kl_beta, ring, graph, schedule=schedule, max_grad_norm=max_grad_norm)
        self.keep_grads = keep_grads

    def _enqueue(self, plan):
        self._train_step(plan, zero_grads=not self.keep_grads)

    def __call__(self, data, eps: Optional[torch.Tensor] = None, next_data=None) -> torch.Tensor:
        return self._run(data, eps, next_data)
