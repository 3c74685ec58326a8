"""Host-side engine: flat parameter storage + the rvae_plan (C ABI) that runs whole steps.

`FlatState` owns the fp32 master weights, gradients, Adam moments, the device step counter and the bf16 shadow
planes in the layout of `rvae_param_layout_padded` (W1 | W2=[fc21;fc22] | W3 | W4 | b1 | b2 | b3 | b4, each block
at the dims rounded up to multiples of 64). The nn.Module parameters are views into it - the top-left corners of their
blocks, strided when a dim is padded - so `state_dict()` stays reference-compatible while one kernel can update
everything.
`Plan` binds those buffers plus a workspace to an rvae_plan for a maximum batch size.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import torch

from . import _lib, ops
from ._lib import check

PRECISIONS = {"bf16": ops.PRECISION_BF16, "fp32": ops.PRECISION_FP32}

# nn.Parameter -> (FlatState, parameter name). Kept OUTSIDE the parameters: torch pickles a Parameter's custom
# attributes, so hanging the FlatState on them would drag gradients, both Adam moments and the bf16 shadows into
# torch.save(model) (best_model.pt / last_model.pt) and make the file unloadable where only the reference's
# rawvae.model exists. Identity-keyed and weak: entries vanish with their parameters.
from torch.utils.weak import WeakTensorKeyDictionary  # noqa: E402

_FLAT_OF = WeakTensorKeyDictionary()


def register_flat(param: torch.Tensor, flat: "FlatState", name: str) -> None:
    _FLAT_OF[param] = (flat, name)


def flat_of(param: torch.Tensor):
    """(FlatState, name) of a parameter that is a view of a flat buffer, else None."""
    return _FLAT_OF.get(param)

# parameter name -> (layout field, row offset factor) ; fc21/fc22 share the stacked W2 / b2 blocks
PARAM_SLOTS = ("fc1.weight", "fc1.bias", "fc21.weight", "fc21.bias", "fc22.weight", "fc22.bias",
               "fc3.weight", "fc3.bias", "fc4.weight", "fc4.bias")


def param_layout(S: int, H: int, L: int) -> _lib.Layout:
    lay = _lib.Layout()
    check(_lib.load().rvae_param_layout(S, H, L, C.byref(lay)))
    return lay


def param_layout_padded(S: int, H: int, L: int) -> Tuple[_lib.Layout, int, int, int]:
    """(layout of the padded blocks, Sp, Hp, Lp): any positive dims, rounded up to multiples of 64."""
    lay, sp, hp, lp = _lib.Layout(), C.c_int(), C.c_int(), C.c_int()
    check(_lib.load().rvae_param_layout_padded(S, H, L, C.byref(lay), C.byref(sp), C.byref(hp), C.byref(lp)))
    return lay, sp.value, hp.value, lp.value


def param_geometry(S: int, H: int, L: int) -> Dict[str, Tuple[int, Tuple[int, ...], Tuple[int, ...]]]:
    """name -> (element offset in the flat buffer, shape, strides): each parameter is the top-left corner of its
    padded block (row pitch = the block's padded width); contiguous when the dims are multiples of 64."""
    lay, Sp, Hp, Lp = param_layout_padded(S, H, L)
    return {
        "fc1.weight": (lay.w1, (H, S), (Sp, 1)), "fc1.bias": (lay.b1, (H,), (1,)),
        "fc21.weight": (lay.w2, (L, H), (Hp, 1)), "fc21.bias": (lay.b2, (L,), (1,)),
        "fc22.weight": (lay.w2 + Lp * Hp, (L, H), (Hp, 1)), "fc22.bias": (lay.b2 + Lp, (L,), (1,)),
        "fc3.weight": (lay.w3, (H, L), (Lp, 1)), "fc3.bias": (lay.b3, (H,), (1,)),
        "fc4.weight": (lay.w4, (S, H), (Hp, 1)), "fc4.bias": (lay.b4, (S,), (1,)),
    }


def param_offsets(S: int, H: int, L: int) -> Dict[str, Tuple[int, Tuple[int, ...]]]:
    """name -> (element offset in the flat buffer, shape)."""
    return {n: (off, shape) for n, (off, shape, _) in param_geometry(S, H, L).items()}


class FlatState:
    def __init__(self, S: int, H: int, L: int, device: torch.device, precision: str = "bf16"):
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
        self.S, self.H, self.L = S, H, L
        self.device = device
        self.precision = precision
        self.geometry = param_geometry(S, H, L)
        self.offsets = {n: (off, shape) for n, (off, shape, _) in self.geometry.items()}
        lay, self.Sp, self.Hp, self.Lp = param_layout_padded(S, H, L)
        self.total = int(lay.total)
        z = lambda dt: torch.zeros(self.total, dtype=dt, device=device)
        self.params = z(torch.float32)
        self.grads = z(torch.float32)
        self.exp_avg = z(torch.float32)
        self.exp_avg_sq = z(torch.float32)
        self.step = torch.zeros((), dtype=torch.float32, device=device)
        self.shadow_hi = z(torch.bfloat16)
        self.shadow_lo = z(torch.bfloat16) if precision == "fp32" else None
        self.shadow_version = -1  # sum of parameter version counters at the last shadow refresh

    def view(self, buf: torch.Tensor, name: str) -> torch.Tensor:
        off, shape, strides = self.geometry[name]
        if len(shape) == 2 and strides[0] != shape[1]:   # a padded block: strided view of its top-left corner
            return buf[off:off + shape[0] * strides[0]].view(shape[0], strides[0])[:, :shape[1]]
        n = 1
        for s in shape:
            n *= s
        return buf[off:off + n].view(shape)

    def sync_shadow(self) -> None:
        lib = _lib.load()
        check(lib.rvae_split_bf16(ops.ctx(self.device), self.params.data_ptr(), self.total,
                                  self.shadow_hi.data_ptr(),
                                  self.shadow_lo.data_ptr() if self.shadow_lo is not None else None,
                                  torch.cuda.current_stream().cuda_stream))


class Plan:
    """rvae_plan bound to a FlatState and a zero-initialised workspace for batches up to `max_batch` frames."""

    def __init__(self, flat: FlatState, max_batch: int):
        lib = _lib.load()
        self.flat = flat
        self.max_batch = int(max_batch)
        self.lib = lib
        self.handle = C.c_void_p()
        with torch.cuda.device(flat.device):
            check(lib.rvae_plan_create(ops.ctx(flat.device), flat.S, flat.H, flat.L, self.max_batch,
                                       PRECISIONS[flat.precision], C.byref(self.handle)))
            nbytes = int(lib.rvae_plan_workspace_bytes(self.handle))
            self.workspace = torch.zeros(nbytes + 256, dtype=torch.uint8, device=flat.device)
            base = self.workspace.data_ptr()
            aligned = (base + 255) // 256 * 256
            bufs = _lib.PlanBuffers(flat.params.data_ptr(), flat.grads.data_ptr(), flat.exp_avg.data_ptr(),
                                    flat.exp_avg_sq.data_ptr(), flat.step.data_ptr(), flat.shadow_hi.data_ptr(),
                                    flat.shadow_lo.data_ptr() if flat.shadow_lo is not None else None, aligned)
            check(lib.rvae_plan_bind(self.handle, C.byref(bufs)))
        self.batch = 0
        self.cur = 0    # which of the two input sets is current (flips with every swap_prefetched)
        self.pitch = 0      # 0: the current input set holds gathered [batch, S] rows; hop: a sample span read in place
        self.pitch_alt = 0  # the same for the prefetched set
        self.token = 0  # bumped whenever a new batch is loaded (activations of older forwards are gone)

    def __del__(self):
        try:
            if self.handle:
                self.lib.rvae_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    @staticmethod
    def _stream() -> int:
        return torch.cuda.current_stream().cuda_stream

    # ---- inputs
    def load_batch(self, x: torch.Tensor) -> None:
        if not x.is_cuda:
            raise _lib.RvaeError("input batch must be a CUDA tensor; there is no CPU fallback")
        x = x.reshape(-1, self.flat.S)
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        check(self.lib.rvae_plan_load_batch(self.handle, x.data_ptr(), x.shape[0], self._stream()))
        self.batch = x.shape[0]
        self.pitch = 0
        self.token += 1

    def span_supported(self, count: int, hop: int) -> bool:
        """Can a run of `count` consecutive frames at stride `hop` be read in place (load_frames(span=True))?"""
        return bool(self.lib.rvae_plan_span_supported(self.handle, int(count), int(hop)))

    def load_frames(self, audio: torch.Tensor, count: int, hop: int, *, frame_idx: Optional[torch.Tensor] = None,
                    first_frame: int = 0, row_offset: int = 0, span: bool = False) -> None:
        """span=True: the frames are the RUN first_frame .. first_frame + count (or frame_idx[0] .., read on the
        device) and are read in place from the converted sample span (rvae_plan_load_span)."""
        if audio.dtype not in (torch.float32, torch.int16) or not audio.is_cuda or not audio.is_contiguous():
            raise _lib.RvaeError("audio must be a contiguous CUDA float32 / int16 tensor")
        if span:
            if row_offset != 0:
                raise _lib.RvaeError("a span batch cannot be appended to")
            if frame_idx is not None and (frame_idx.dtype != torch.int64 or not frame_idx.is_cuda or frame_idx.numel() < 1):
                raise _lib.RvaeError("frame_idx must be a CUDA int64 tensor whose first entry is the run's first frame")
            check(self.lib.rvae_plan_load_span(self.handle, audio.data_ptr(), int(audio.dtype == torch.int16),
                                               audio.numel(), frame_idx.data_ptr() if frame_idx is not None else None,
                                               first_frame, count, hop, self._stream()))
            self.batch, self.pitch = count, hop
            self.token += 1
            return
        if frame_idx is not None and (frame_idx.dtype != torch.int64 or not frame_idx.is_cuda
                                      or frame_idx.numel() != count or not frame_idx.is_contiguous()):
            raise _lib.RvaeError("frame_idx must be a contiguous CUDA int64 tensor with `count` entries")
        check(self.lib.rvae_plan_load_frames(self.handle, audio.data_ptr(), int(audio.dtype == torch.int16),
                                             audio.numel(), frame_idx.data_ptr() if frame_idx is not None else None,
                                             first_frame, count, hop, row_offset, self._stream()))
        self.batch = row_offset + count
        self.pitch = 0
        if row_offset == 0:
            self.token += 1

    def prefetch_frames(self, audio: torch.Tensor, count: int, hop: int, *, frame_idx: Optional[torch.Tensor] = None,
                        first_frame: int = 0, seed: int = 0, offset: int = 0, add_step: bool = True,
                        span: bool = False) -> None:
        """Describe the NEXT step's batch: the next train_step gathers it (and draws its noise) in the background.
        span=True: a run of consecutive frames, read in place (see load_frames)."""
        if audio.dtype not in (torch.float32, torch.int16) or not audio.is_cuda or not audio.is_contiguous():
            raise _lib.RvaeError("audio must be a contiguous CUDA float32 / int16 tensor")
        if span:
            if frame_idx is not None and (frame_idx.dtype != torch.int64 or not frame_idx.is_cuda or frame_idx.numel() < 1):
                raise _lib.RvaeError("frame_idx must be a CUDA int64 tensor whose first entry is the run's first frame")
            check(self.lib.rvae_plan_prefetch_span(self.handle, audio.data_ptr(), int(audio.dtype == torch.int16),
                                                   audio.numel(), frame_idx.data_ptr() if frame_idx is not None else None,
                                                   first_frame, count, hop, seed, offset, int(add_step)))
            self.pitch_alt = hop
            return
        self.pitch_alt = 0
        if frame_idx is not None and (frame_idx.dtype != torch.int64 or not frame_idx.is_cuda
                                      or frame_idx.numel() != count or not frame_idx.is_contiguous()):
            raise _lib.RvaeError("frame_idx must be a contiguous CUDA int64 tensor with `count` entries")
        check(self.lib.rvae_plan_prefetch_frames(self.handle, audio.data_ptr(), int(audio.dtype == torch.int16),
                                                 audio.numel(), frame_idx.data_ptr() if frame_idx is not None else None,
                                                 first_frame, count, hop, seed, offset, int(add_step)))

    def prefetched_batch(self) -> int:
        return int(self.lib.rvae_plan_prefetched_batch(self.handle))

    def swap_prefetched(self) -> None:
        """Make the prefetched batch (and its noise) the current one - replaces load_frames + gen_eps."""
        n = self.prefetched_batch()
        check(self.lib.rvae_plan_swap_prefetched(self.handle))
        self.batch = n
        self.cur ^= 1
        self.pitch, self.pitch_alt = self.pitch_alt, self.pitch
        self.token += 1

    def join_background(self) -> None:
        """The current stream waits for pending background work of earlier calls (needed before a graph capture)."""
        check(self.lib.rvae_plan_join_background(self.handle, self._stream()))

    def note_prefetched(self, count: int, span_hop: int = 0) -> None:
        """A replayed CUDA graph gathered `count` frames into the alternate input set (span_hop > 0: as a sample span
        read in place at that pitch): record it on the host side."""
        check(self.lib.rvae_plan_note_prefetched(self.handle, count, span_hop))
        self.pitch_alt = span_hop

    def set_eps(self, eps: torch.Tensor) -> None:
        if eps.dtype != torch.float32 or not eps.is_cuda or not eps.is_contiguous():
            eps = eps.to(device=self.flat.device, dtype=torch.float32).contiguous()
        if eps.numel() != self.batch * self.flat.L:
            raise _lib.RvaeError(f"eps has {eps.numel()} elements, expected {self.batch}x{self.flat.L}")
        check(self.lib.rvae_plan_set_eps(self.handle, eps.data_ptr(), self._stream()))

    def gen_eps(self, seed: int, offset: int, add_step: bool = False) -> None:
        check(self.lib.rvae_plan_gen_eps(self.handle, seed, offset, int(add_step), self._stream()))

    def set_outputs(self, mu=None, logvar=None, xhat=None) -> None:
        p = lambda t: t.data_ptr() if t is not None else None
        check(self.lib.rvae_plan_set_outputs(self.handle, p(mu), p(logvar), p(xhat)))

    def enable_dp(self, on: bool = True) -> None:
        check(self.lib.rvae_plan_enable_dp(self.handle, int(on)))

    def set_noise_rows(self, first_global_row: int) -> None:
        """Data parallelism: this rank's shard starts at row `first_global_row` of the global batch (Philox counters
        of gen_eps / prefetch_frames start there, so equal seeds give the single-process noise on every rank)."""
        check(self.lib.rvae_plan_set_noise_rows(self.handle, int(first_global_row)))

    def set_global_batch(self, global_batch: int) -> None:
        check(self.lib.rvae_plan_set_global_batch(self.handle, int(global_batch)))

    # ---- steps
    def forward(self, kl_beta: float, fused_loss: bool, want_xhat: bool) -> None:
        check(self.lib.rvae_plan_forward(self.handle, kl_beta, int(fused_loss), int(want_xhat), self._stream()))

    def backward(self, stage: int = -1) -> None:
        check(self.lib.rvae_plan_backward(self.handle, stage, self._stream()))

    def backward_external(self, g_xhat, xhat, g_mu, g_logvar, logvar) -> None:
        check(self.lib.rvae_plan_backward_external(self.handle, g_xhat.data_ptr(), xhat.data_ptr(), g_mu.data_ptr(),
                                                   g_logvar.data_ptr(), logvar.data_ptr(), self._stream()))

    def finish_loss(self, kl_beta: float, loss_out: Optional[torch.Tensor], ring_size: int = 1) -> None:
        check(self.lib.rvae_plan_finish_loss(self.handle, kl_beta,
                                             loss_out.data_ptr() if loss_out is not None else None, ring_size,
                                             self._stream()))

    def finish_loss_deferred(self, kl_beta: float, loss_out: Optional[torch.Tensor], ring_size: int = 1) -> None:
        """Like finish_loss, but carried out by the latent backward kernel of the next backward stage 1 (no launch)."""
        check(self.lib.rvae_plan_finish_loss_deferred(self.handle, kl_beta,
                                                      loss_out.data_ptr() if loss_out is not None else None, ring_size))

    def adam_buckets(self, mask: int, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, grad_scale=1.0,
                     zero_grads=False) -> None:
        """Adam over the gradient buckets in `mask` (bit s = bucket s; 0..3 = W4, W3, W2, W1, 4 = biases)."""
        check(self.lib.rvae_plan_adam_buckets(self.handle, mask, lr, beta1, beta2, eps, weight_decay, grad_scale,
                                              int(zero_grads), self._stream()))

    def adam(self, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, grad_scale=1.0, zero_grads=False) -> None:
        check(self.lib.rvae_plan_adam(self.handle, lr, beta1, beta2, eps, weight_decay, grad_scale, int(zero_grads),
                                      self._stream()))

    def train_step(self, kl_beta, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0,
                   loss_out: Optional[torch.Tensor] = None, ring_size: int = 1, zero_grads: bool = True) -> None:
        check(self.lib.rvae_plan_train_step(self.handle, kl_beta, lr, beta1, beta2, eps, weight_decay, int(zero_grads),
                                            loss_out.data_ptr() if loss_out is not None else None, ring_size,
                                            self._stream()))

    def train_step_hp(self, hp: torch.Tensor, loss_out: Optional[torch.Tensor] = None, ring_size: int = 1,
                      zero_grads: bool = True) -> None:
        """train_step with every hyper-parameter read from the device record `hp` (schedule.Schedule) when the
        kernels run: a captured graph of this call follows the schedule and any rewrite of the record."""
        check(self.lib.rvae_plan_train_step_hp(self.handle, hp.data_ptr(), int(zero_grads),
                                               loss_out.data_ptr() if loss_out is not None else None, ring_size,
                                               self._stream()))

    def set_grad_clip(self, max_norm_ptr: Optional[int], norm_out: Optional[torch.Tensor] = None,
                      ring_size: int = 1) -> None:
        """Clip the gradient of every later training step by its global norm at the device double max_norm_ptr
        (None = off); the pre-clip norm of each step goes to norm_out[step mod ring_size] when norm_out is given."""
        check(self.lib.rvae_plan_set_grad_clip(self.handle, max_norm_ptr,
                                               norm_out.data_ptr() if norm_out is not None else None, int(ring_size)))

    def set_ema(self, ema: Optional[torch.Tensor], decay_ptr: Optional[int] = None,
                n_averaged: Optional[torch.Tensor] = None) -> None:
        """Update the fp32 EMA buffer `ema` (the flat layout of the parameters) in every Adam launch of every later
        training step, with the device double decay at decay_ptr and the device int64 count n_averaged (None = off)."""
        if ema is None:
            check(self.lib.rvae_plan_set_ema(self.handle, None, None, None))
            return
        if ema.dtype != torch.float32 or ema.numel() != self.flat.total or ema.device != self.flat.device:
            raise _lib.RvaeError("the EMA buffer must be a float32 tensor of the flat parameter layout")
        if n_averaged is None or n_averaged.dtype != torch.int64 or n_averaged.device != self.flat.device:
            raise _lib.RvaeError("n_averaged must be an int64 tensor on the plan's device")
        check(self.lib.rvae_plan_set_ema(self.handle, ema.data_ptr(), decay_ptr, n_averaged.data_ptr()))

    def deterministic_bytes(self) -> int:
        """Scratch bytes of the deterministic training step at this plan's max_batch (rvae_plan_deterministic_bytes)."""
        return int(self.lib.rvae_plan_deterministic_bytes(self.handle))

    def set_deterministic(self, on: bool) -> None:
        """Make this plan's training steps bitwise reproducible (on) or use the default kernels (off). The scratch is
        allocated on first use and kept with the plan, so a captured graph's addresses stay valid."""
        if not on:
            check(self.lib.rvae_plan_set_deterministic(self.handle, None, 0))
            return
        scratch = getattr(self, "_det_scratch", None)
        if scratch is None:
            nbytes = self.deterministic_bytes()
            scratch = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.flat.device)
            self._det_scratch = scratch
        aligned = (scratch.data_ptr() + 255) // 256 * 256
        check(self.lib.rvae_plan_set_deterministic(self.handle, aligned, scratch.numel() - (aligned - scratch.data_ptr())))

    def grad_norm(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Global L2 norm of the bound gradient buffer, with the kernels of a clipping step (0-dim float32 tensor)."""
        if out is None:
            out = torch.empty((), dtype=torch.float32, device=self.flat.device)
        check(self.lib.rvae_plan_grad_norm(self.handle, out.data_ptr(), self._stream()))
        return out

    def encode(self) -> None:
        check(self.lib.rvae_plan_encode(self.handle, self._stream()))

    def decode(self, z: torch.Tensor, xhat_out: torch.Tensor) -> None:
        check(self.lib.rvae_plan_decode(self.handle, z.data_ptr(), z.shape[0], xhat_out.data_ptr(), self._stream()))
        self.batch = z.shape[0]
        self.token += 1

    def decode_lerp(self, mu_a, lv_a, mu_b, lv_b, alpha, eps, xhat_out) -> None:
        """lerp(alpha per frame) -> reparameterize -> decode as one chained enqueue (tutorial.ipynb:496-510, 905-932)."""
        n = mu_a.shape[0]
        check(self.lib.rvae_plan_decode_lerp(self.handle, mu_a.data_ptr(), lv_a.data_ptr(), mu_b.data_ptr(),
                                             lv_b.data_ptr(), alpha.data_ptr(), int(alpha.dtype == torch.float64),
                                             eps.data_ptr() if eps is not None else None, n, xhat_out.data_ptr(),
                                             self._stream()))
        self.batch = n
        self.token += 1

    GEMM_SLOTS = ("F1", "F2", "F3", "F4_out", "F4_lin", "B4w", "B4d", "B3w", "B3d", "B2w", "B2d", "B1w")
    AUX_SLOTS = ("load", "eps", "finalize", "colsum", "adam", "tanh_bwd", "latent_bwd")

    def enable_timing(self, on: bool) -> None:
        check(self.lib.rvae_plan_enable_timing(self.handle, int(on)))

    def read_timing(self):
        """{slot: (total_ms, launches, flops_per_launch)} since the last read (synchronises the timing events)."""
        names = self.GEMM_SLOTS + self.AUX_SLOTS
        n = len(names)
        ms, cnt, fl = (C.c_float * n)(), (C.c_int64 * n)(), (C.c_double * n)()
        check(self.lib.rvae_plan_read_timing(self.handle, ms, cnt, fl))
        return {k: (float(ms[i]), int(cnt[i]), float(fl[i])) for i, k in enumerate(names)}

    ACTIVATIONS = ("x", "h1", "z", "h3", "da4", "da3", "d_ml", "da1")

    def activation(self, name: str):
        """(hi, lo) bf16 views [batch, cols] of an intermediate of the current batch (lo is None in bf16 mode).
        Introspection for tests / debugging; the tensors alias the workspace and are overwritten by the next step."""
        hi, lo, cols = C.c_void_p(), C.c_void_p(), C.c_int()
        check(self.lib.rvae_plan_activation(self.handle, self.ACTIVATIONS.index(name), C.byref(hi), C.byref(lo),
                                            C.byref(cols)))

        def view(ptr):
            if not ptr:
                return None
            off = ptr - self.workspace.data_ptr()
            n = self.batch * cols.value
            return self.workspace[off:off + 2 * n].view(torch.bfloat16).view(self.batch, cols.value)
        return view(hi.value), view(lo.value)

    def latent(self, name: str) -> torch.Tensor:
        """fp32 view [batch, L] of the current batch's `eps` (the noise the step used - Philox or injected), `mu` or
        `logvar` in the workspace. Introspection for tests: aliases the workspace, overwritten by the next step.
        (A strided view when latent_dim is padded: the workspace rows are Lp wide.)"""
        fn = {"eps": self.lib.rvae_plan_eps, "mu": self.lib.rvae_plan_mu, "logvar": self.lib.rvae_plan_logvar}[name]
        return self._rows(int(fn(self.handle)), self.flat.L, self.flat.Lp)

    def xhat(self) -> torch.Tensor:
        """fp32 view [batch, S] of the current batch's xhat in the workspace (after a forward that left xhat there:
        set_outputs without an xhat tensor). Aliases the workspace; rows are Sp wide when segment_length is padded."""
        return self._rows(int(self.lib.rvae_plan_xhat(self.handle)), self.flat.S, self.flat.Sp)

    def _rows(self, ptr: int, cols: int, pitch: int) -> torch.Tensor:
        off = ptr - self.workspace.data_ptr()
        n = self.batch * pitch
        return self.workspace[off:off + 4 * n].view(torch.float32).view(self.batch, pitch)[:, :cols]

    def bucket(self, s: int) -> torch.Tensor:
        """Gradient bucket s as a view of flat.grads (0..3 = W4, W3, W2, W1 in backward order; 4 = biases)."""
        ptr, cnt = C.c_void_p(), C.c_int64()
        check(self.lib.rvae_plan_bucket(self.handle, s, C.byref(ptr), C.byref(cnt)))
        off = (ptr.value - self.flat.grads.data_ptr()) // 4
        return self.flat.grads[off:off + cnt.value]
