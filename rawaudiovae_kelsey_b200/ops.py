"""Tensor-level wrappers over the C ABI. PyTorch is only the allocator / stream provider here: every function
checks its tensors (CUDA, contiguous, dtype), then passes raw device pointers and the current CUDA stream to
librvae_b200. CPU tensors raise - there is no CPU fallback on the product path.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import check

ACT_NONE, ACT_RELU, ACT_TANH, ACT_TANH_APPROX = 0, 1, 2, 3
PRECISION_BF16, PRECISION_FP32 = 0, 1

_CTX = {}


def _require_cuda() -> None:
    if not torch.cuda.is_available():
        raise _lib.RvaeError("rawaudiovae_kelsey_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def ctx(device: Optional[torch.device] = None) -> int:
    """Per-device rvae_ctx handle (created on first use)."""
    _require_cuda()
    idx = torch.cuda.current_device() if device is None or device.index is None else device.index
    h = _CTX.get(idx)
    if h is None:
        lib = _lib.load()
        out = C.c_void_p()
        with torch.cuda.device(idx):
            torch.cuda.init()
            torch.zeros(1, device=f"cuda:{idx}")  # make sure the primary context exists
            check(lib.rvae_ctx_create(idx, C.byref(out)))
        h = out.value
        _CTX[idx] = h
    return h


def launch_count(device: Optional[torch.device] = None) -> int:
    return int(_lib.load().rvae_ctx_launch_count(ctx(device)))


def num_sms(device: Optional[torch.device] = None) -> int:
    return int(_lib.load().rvae_ctx_num_sms(ctx(device)))


TRACE_HEADER, TRACE_TILES, TRACE_EVENTS = 16, 24, 16
TRACE_WORDS_PER_CTA = TRACE_HEADER + TRACE_TILES * TRACE_EVENTS


def set_trace(buf: Optional[torch.Tensor], launches: int = 1) -> None:
    """Debug: direct the GEMM timeline trace (csrc/gemm.cuh) into an int64 CUDA tensor of
    launches * TRACE_WORDS_PER_CTA * num_sms words (successive GEMM launches fill successive slabs), or switch it
    off with None."""
    if buf is not None and (buf.dtype != torch.int64 or not buf.is_cuda or not buf.is_contiguous()):
        raise _lib.RvaeError("trace buffer must be a contiguous int64 CUDA tensor")
    if buf is not None and buf.numel() < launches * TRACE_WORDS_PER_CTA * num_sms(buf.device):
        raise _lib.RvaeError("trace buffer too small")
    check(_lib.load().rvae_debug_set_trace(ctx(None if buf is None else buf.device),
                                           None if buf is None else buf.data_ptr(), launches))


def set_aux_trace(buf: Optional[torch.Tensor], launches: int = 0) -> None:
    """Debug: trace of the HBM-bound kernels into an int64 CUDA tensor [launches, 8] (column 0 initialised to a large
    value by the caller: it is reduced with atomicMin), or off with None."""
    check(_lib.load().rvae_debug_set_aux_trace(ctx(None if buf is None else buf.device),
                                               None if buf is None else buf.data_ptr(), launches))


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor], dtype: Optional[torch.dtype] = None, name: str = "tensor") -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.RvaeError(f"{name} must be a CUDA tensor (got {t.device}); there is no CPU fallback")
    if not t.is_contiguous():
        raise _lib.RvaeError(f"{name} must be contiguous")
    if dtype is not None and t.dtype != dtype:
        raise _lib.RvaeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.data_ptr()


def _planes(t, name):
    """A bf16 operand is either a bf16 tensor or a (hi, lo) tuple of bf16 tensors."""
    if isinstance(t, (tuple, list)):
        hi, lo = t
        return _ptr(hi, torch.bfloat16, name + ".hi"), _ptr(lo, torch.bfloat16, name + ".lo")
    return _ptr(t, torch.bfloat16, name), None


# --------------------------------------------------------------------------------------------- framing
def frame_gather(audio: torch.Tensor, n_frames: int, hop: int, S: int, *, frame_idx: Optional[torch.Tensor] = None,
                 first_frame: int = 0, out_f32: bool = True, out_bf16: bool = False, out_lo: bool = False):
    """Slice a device-resident wav buffer (float32 or int16) into [n_frames, S] frames on the GPU.
    Returns (f32 or None, bf16_hi or None, bf16_lo or None)."""
    lib = _lib.load()
    if audio.dtype not in (torch.float32, torch.int16):
        raise _lib.RvaeError("audio must be float32 or int16")
    a = _ptr(audio, None, "audio")
    dev = audio.device
    f32 = torch.empty((n_frames, S), dtype=torch.float32, device=dev) if out_f32 else None
    hi = torch.empty((n_frames, S), dtype=torch.bfloat16, device=dev) if out_bf16 else None
    lo = torch.empty((n_frames, S), dtype=torch.bfloat16, device=dev) if (out_bf16 and out_lo) else None
    if frame_idx is not None and frame_idx.numel() != n_frames:
        raise _lib.RvaeError("frame_idx must have n_frames entries")
    check(lib.rvae_frame_gather(ctx(dev), a, int(audio.dtype == torch.int16), audio.numel(),
                                _ptr(frame_idx, torch.int64, "frame_idx"), first_frame, n_frames, hop, S,
                                _ptr(hi), _ptr(lo), _ptr(f32), _stream()))
    return f32, hi, lo


def overlap_add(frames: torch.Tensor, hop: int, n_out: Optional[int] = None, *, t_begin: int = 0,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[t - t_begin] = overlap-add of `frames` (fp32 [n, S], cut at stride hop) at sample t, for n_out samples from
    t_begin on (default: the whole signal). `out`: write into this 1-D fp32 tensor instead of allocating."""
    lib = _lib.load()
    n_frames, S = frames.shape
    if n_out is None:
        n_out = out.numel() if out is not None else max((n_frames - 1) * hop + S - t_begin, 0) if n_frames > 0 else 0
    if out is None:
        out = torch.empty((n_out,), dtype=torch.float32, device=frames.device)
    elif out.numel() < n_out:
        raise _lib.RvaeError("overlap_add: output tensor too small")
    check(lib.rvae_overlap_add(ctx(frames.device), _ptr(frames, torch.float32, "frames"), n_frames, S, hop,
                               _ptr(out, torch.float32, "out"), t_begin, n_out, _stream()))
    return out


# --------------------------------------------------------------------------------------------- elementwise
def randn(shape, seed: int, offset: int = 0, device=None, elem_base: int = 0) -> torch.Tensor:
    """eps ~ N(0,1) from Philox (seed, offset); `elem_base` (any value >= 0) makes the result elements
    [elem_base, elem_base + n) of the logical noise tensor - a rank's rows of a global batch."""
    lib = _lib.load()
    out = torch.empty(shape, dtype=torch.float32, device=device or "cuda")
    check(lib.rvae_randn(ctx(out.device), _ptr(out), out.numel(), seed, offset, elem_base, _stream()))
    return out


def lerp_reparameterize(mu_a, logvar_a, mu_b, logvar_b, alpha, eps=None, *, want_z=True, want_dist=False):
    """Per-frame latent interpolation + reparameterisation (tutorial.ipynb:496-510, 905-932).
    alpha: [rows] float32 or float64 CUDA tensor. Returns (z or None, mu or None, logvar or None), fp32 [rows, L]."""
    lib = _lib.load()
    rows, L = mu_a.shape
    if alpha.dtype not in (torch.float32, torch.float64) or alpha.numel() != rows:
        raise _lib.RvaeError("alpha must be a float32 / float64 tensor with one entry per frame")
    dev = mu_a.device
    f = lambda on: torch.empty((rows, L), dtype=torch.float32, device=dev) if on else None
    z, mu, lv = f(want_z), f(want_dist), f(want_dist)
    check(lib.rvae_lerp_reparameterize(ctx(dev), _ptr(mu_a, torch.float32, "mu_a"), _ptr(logvar_a, torch.float32, "logvar_a"),
                                       _ptr(mu_b, torch.float32, "mu_b"), _ptr(logvar_b, torch.float32, "logvar_b"),
                                       _ptr(alpha, None, "alpha"), int(alpha.dtype == torch.float64),
                                       _ptr(eps, torch.float32, "eps"), rows, L, _ptr(z), _ptr(mu), _ptr(lv), _stream()))
    return z, mu, lv


def split_bf16(src: torch.Tensor, want_lo: bool = False) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    lib = _lib.load()
    hi = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    lo = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device) if want_lo else None
    check(lib.rvae_split_bf16(ctx(src.device), _ptr(src, torch.float32, "src"), src.numel(), _ptr(hi), _ptr(lo),
                              _stream()))
    return hi, lo


def reparameterize(mu: torch.Tensor, logvar: torch.Tensor, eps: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    z = torch.empty_like(mu)
    check(lib.rvae_reparameterize(ctx(mu.device), _ptr(mu, torch.float32, "mu"), _ptr(logvar, torch.float32, "logvar"),
                                  _ptr(eps, torch.float32, "eps"), mu.numel(), _ptr(z), _stream()))
    return z


def loss_fwd(xhat, x, mu, logvar, beta: float) -> torch.Tensor:
    lib = _lib.load()
    B, S = xhat.shape
    L = mu.shape[1]
    acc = torch.zeros(2, dtype=torch.float64, device=xhat.device)
    out = torch.empty((), dtype=torch.float32, device=xhat.device)
    check(lib.rvae_loss_fwd(ctx(xhat.device), _ptr(xhat, torch.float32, "xhat"), _ptr(x, torch.float32, "x"),
                            _ptr(mu, torch.float32, "mu"), _ptr(logvar, torch.float32, "logvar"), B, S, L, beta,
                            _ptr(acc), _ptr(out), _stream()))
    return out


def _rows(t: torch.Tensor, name: str) -> Tuple[int, int]:
    """(data pointer, row pitch) of an fp32 CUDA matrix whose rows are contiguous (a strided row view is fine)."""
    if not t.is_cuda or t.dtype != torch.float32 or t.dim() != 2:
        raise _lib.RvaeError(f"{name} must be a 2-D float32 CUDA tensor")
    if t.shape[1] > 1 and t.stride(1) != 1:
        raise _lib.RvaeError(f"{name} must have contiguous rows")
    return t.data_ptr(), max(t.stride(0), t.shape[1])


def frame_loss(xhat: torch.Tensor, mu: torch.Tensor, logvar: torch.Tensor, audio: torch.Tensor, first_frame: int,
               hop: int, rec: Optional[torch.Tensor] = None, kl: Optional[torch.Tensor] = None
               ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per-frame reconstruction and KL terms (rvae_frame_loss) of the frames first_frame, first_frame + 1, ... of the
    wav buffer `audio` (float32 / int16), cut at stride hop: rec[f] = mean_s (xhat[f] - x[f])^2,
    kl[f] = -0.5 * mean_l (1 + logvar - mu^2 - exp(logvar)). xhat [rows, S], mu / logvar [rows, L] may be row views
    of wider buffers (a plan's workspace). Returns (rec, kl), fp32 [rows] (written into `rec` / `kl` if given)."""
    lib = _lib.load()
    if audio.dtype not in (torch.float32, torch.int16) or audio.dim() != 1:
        raise _lib.RvaeError("audio must be a 1-D float32 or int16 tensor")
    px, ldx = _rows(xhat, "xhat")
    pm, ldm = _rows(mu, "mu")
    pl, ldl = _rows(logvar, "logvar")
    rows, S = xhat.shape
    L = mu.shape[1]
    if mu.shape != logvar.shape or mu.shape[0] != rows:
        raise _lib.RvaeError("mu and logvar must be [rows, L] with the rows of xhat")
    if ldm != ldl:
        raise _lib.RvaeError("mu and logvar must share one row pitch")
    dev = xhat.device
    rec = torch.empty(rows, dtype=torch.float32, device=dev) if rec is None else rec
    kl = torch.empty(rows, dtype=torch.float32, device=dev) if kl is None else kl
    if rec.numel() != rows or kl.numel() != rows:
        raise _lib.RvaeError("rec and kl must hold one value per frame")
    if any(t.device != dev for t in (mu, logvar, audio, rec, kl)):
        raise _lib.RvaeError("xhat, mu, logvar, audio, rec and kl must be on one device")
    check(lib.rvae_frame_loss(ctx(dev), px, ldx, pm, pl, ldm, rows, S, L, _ptr(audio, None, "audio"),
                              int(audio.dtype == torch.int16), audio.numel(), int(first_frame), int(hop),
                              _ptr(rec, torch.float32, "rec"), _ptr(kl, torch.float32, "kl"), _stream()))
    return rec, kl


def hparams_eval(record: torch.Tensor, k: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Evaluate the schedule of a device rvae_hparams record (schedule.DeviceRecord.tensor) at the step indices k
    (int64) with the device function of the training kernels. Returns (lr float64, beta float32), shaped like k."""
    lib = _lib.load()
    if record.dtype != torch.uint8 or record.numel() != C.sizeof(_lib.Hparams) or not record.is_cuda:
        raise _lib.RvaeError("record must be a CUDA uint8 tensor of sizeof(rvae_hparams) bytes")
    if k.dtype != torch.int64 or k.device != record.device:
        raise _lib.RvaeError("k must be an int64 tensor on the record's device")
    kc = k.contiguous()
    lr = torch.empty(k.shape, dtype=torch.float64, device=k.device)
    beta = torch.empty(k.shape, dtype=torch.float32, device=k.device)
    check(lib.rvae_hparams_eval(ctx(k.device), record.data_ptr(), kc.data_ptr(), kc.numel(), lr.data_ptr(),
                                beta.data_ptr(), _stream()))
    return lr, beta


def loss_bwd(xhat, x, mu, logvar, beta: float, grad_out: Optional[torch.Tensor]):
    lib = _lib.load()
    B, S = xhat.shape
    L = mu.shape[1]
    g_x = torch.empty_like(xhat)
    g_mu = torch.empty_like(mu)
    g_lv = torch.empty_like(logvar)
    check(lib.rvae_loss_bwd(ctx(xhat.device), _ptr(xhat, torch.float32), _ptr(x, torch.float32),
                            _ptr(mu, torch.float32), _ptr(logvar, torch.float32), B, S, L, beta,
                            _ptr(grad_out, torch.float32, "grad_out"), _ptr(g_x), _ptr(g_mu), _ptr(g_lv), _stream()))
    return g_x, g_mu, g_lv


def tanh_bwd(g_xhat, xhat, want_lo: bool = False):
    lib = _lib.load()
    hi = torch.empty(xhat.shape, dtype=torch.bfloat16, device=xhat.device)
    lo = torch.empty_like(hi) if want_lo else None
    check(lib.rvae_tanh_bwd(ctx(xhat.device), _ptr(g_xhat, torch.float32), _ptr(xhat, torch.float32), xhat.numel(),
                            _ptr(hi), _ptr(lo), _stream()))
    return hi, lo


def colsum(a, out: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    lib = _lib.load()
    hi, lo = _planes(a, "a")
    t = a[0] if isinstance(a, (tuple, list)) else a
    M, N = t.shape
    if out is None:
        out = torch.zeros((N,), dtype=torch.float32, device=t.device)
        accumulate = True
    check(lib.rvae_colsum(ctx(t.device), hi, lo, M, N, N, _ptr(out, torch.float32), int(accumulate), _stream()))
    return out


def adam_step(p, g, m, v, step, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, grad_scale=1.0,
              shadow_hi=None, shadow_lo=None, increment_step: bool = True) -> None:
    """One fused Adam step over flat fp32 buffers. `step` is a device fp32 scalar tensor (torch's state format)."""
    lib = _lib.load()
    c = ctx(p.device)
    if increment_step:
        check(lib.rvae_step_inc(c, _ptr(step, torch.float32, "step"), _stream()))
    check(lib.rvae_adam_step(c, _ptr(p, torch.float32, "p"), _ptr(g, torch.float32, "g"), _ptr(m, torch.float32, "m"),
                             _ptr(v, torch.float32, "v"), p.numel(), lr, beta1, beta2, eps, weight_decay, grad_scale,
                             _ptr(step, torch.float32, "step"), _ptr(shadow_hi, torch.bfloat16),
                             _ptr(shadow_lo, torch.bfloat16), _stream()))


def ema_update(ema: torch.Tensor, params: torch.Tensor, decay: torch.Tensor, n_averaged: torch.Tensor) -> None:
    """ema = lerp(ema, params, 1 - decay) in place (a copy when n_averaged == 0), then n_averaged += 1: one launch
    over flat fp32 buffers. decay: a device float64 scalar tensor, n_averaged a device int64 one."""
    if ema.numel() != params.numel():
        raise _lib.RvaeError(f"ema has {ema.numel()} elements, params {params.numel()}")
    check(_lib.load().rvae_ema_update(ctx(ema.device), _ptr(ema, torch.float32, "ema"),
                                      _ptr(params, torch.float32, "params"), ema.numel(),
                                      _ptr(decay, torch.float64, "decay"), _ptr(n_averaged, torch.int64, "n_averaged"),
                                      _stream()))


def histogram_record_layout(n_segs: int, n_edges: int) -> dict:
    """Byte offsets of the fields of an rvae_param_histogram record (include/rvae_b200.h); "bytes" = results only,
    "total" = results + the kernel's scratch (what the device buffer must hold)."""
    nb = n_edges - 1
    a = (4 * n_segs * nb + 7) // 8 * 8
    total = int(_lib.load().rvae_param_histogram_bytes(n_segs, n_edges))
    if total == 0:
        raise _lib.RvaeError(f"param_histogram: {n_segs} segments / {n_edges} edges are not supported")
    return {"counts": 0, "sum": a, "sum_squares": a + 8 * n_segs, "num": a + 16 * n_segs, "min": a + 24 * n_segs,
            "max": a + 28 * n_segs, "bytes": a + 32 * n_segs, "total": total}


def param_histogram(params: torch.Tensor, seg_offsets, seg_lengths, edges, out: Optional[torch.Tensor] = None, *,
                    seg_rows=None, seg_pitch=None):
    """TensorBoard histograms (make_histogram semantics) of the segments params[seg_offsets[s] : + seg_lengths[s]] of
    a flat fp32 CUDA tensor against the float64 bin edges `edges`, in one launch on the current stream. Returns the
    device record (uint8; `out` if given, at least histogram_record_layout(...)["total"] bytes): unpack a host copy
    of its first ["bytes"] bytes with unpack_histogram_record.
    seg_rows / seg_pitch (given together): segment s is seg_rows[s] rows of seg_lengths[s] values, row r starting at
    seg_offsets[s] + r * seg_pitch[s] (a parameter inside the padded block of a padded model)."""
    lib = _lib.load()
    p = _ptr(params, torch.float32, "params")
    offs = np.ascontiguousarray(seg_offsets, dtype=np.int64)
    lens = np.ascontiguousarray(seg_lengths, dtype=np.int64)
    e = np.ascontiguousarray(edges, dtype=np.float64)
    if offs.shape != lens.shape or offs.ndim != 1:
        raise _lib.RvaeError("param_histogram: seg_offsets and seg_lengths must be 1-D and of equal length")
    if (seg_rows is None) != (seg_pitch is None):
        raise _lib.RvaeError("param_histogram: seg_rows and seg_pitch come together")
    rows = np.ones_like(offs) if seg_rows is None else np.ascontiguousarray(seg_rows, dtype=np.int64)
    pitch = lens if seg_pitch is None else np.ascontiguousarray(seg_pitch, dtype=np.int64)
    if rows.shape != offs.shape or pitch.shape != offs.shape:
        raise _lib.RvaeError("param_histogram: seg_rows and seg_pitch must match seg_offsets")
    if offs.size and (int((offs + (rows - 1) * pitch + lens).max()) > params.numel() or int(offs.min()) < 0):
        raise _lib.RvaeError("param_histogram: a segment lies outside params")
    lay = histogram_record_layout(offs.size, e.size)
    if out is None:
        out = torch.empty(lay["total"], dtype=torch.uint8, device=params.device)
    elif out.numel() < lay["total"]:
        raise _lib.RvaeError(f"param_histogram: record buffer holds {out.numel()} bytes, needs {lay['total']}")
    if seg_rows is None:
        check(lib.rvae_param_histogram(ctx(params.device), p, offs.ctypes.data,
                                       lens.ctypes.data, offs.size, e.ctypes.data, e.size, _ptr(out, torch.uint8, "out"),
                                       _stream()))
    else:
        check(lib.rvae_param_histogram_rows(ctx(params.device), p, offs.ctypes.data, rows.ctypes.data, lens.ctypes.data,
                                            pitch.ctypes.data, offs.size, e.ctypes.data, e.size,
                                            _ptr(out, torch.uint8, "out"), _stream()))
    return out


def unpack_histogram_record(buf, n_segs: int, n_edges: int) -> dict:
    """numpy views of a host copy (uint8 tensor or array, at least ["bytes"] long) of a param_histogram record:
    counts int32 [n_segs, n_edges - 1], sum / sum_squares float64, num int64, min / max float32, each [n_segs]."""
    lay = histogram_record_layout(n_segs, n_edges)
    raw = buf.numpy() if isinstance(buf, torch.Tensor) else np.asarray(buf)
    raw = raw[:lay["bytes"]]
    f = lambda key, dt, n: np.frombuffer(raw, dtype=dt, count=n, offset=lay[key])
    return {"counts": f("counts", np.int32, n_segs * (n_edges - 1)).reshape(n_segs, n_edges - 1),
            "sum": f("sum", np.float64, n_segs), "sum_squares": f("sum_squares", np.float64, n_segs),
            "num": f("num", np.int64, n_segs), "min": f("min", np.float32, n_segs), "max": f("max", np.float32, n_segs)}


# --------------------------------------------------------------------------------------------- GEMM-level ops
def linear_act_fwd(x, w, bias, act: int, *, out_bf16=True, out_lo=False, out_f32=False):
    """y = act(x @ w.T + bias). x: bf16 [M,K] or (hi, lo); w: bf16 [N,K] or (hi, lo)."""
    lib = _lib.load()
    xh, xl = _planes(x, "x")
    wh, wl = _planes(w, "w")
    xt = x[0] if isinstance(x, (tuple, list)) else x
    wt = w[0] if isinstance(w, (tuple, list)) else w
    M, K = xt.shape
    N = wt.shape[0]
    dev = xt.device
    y_hi = torch.empty((M, N), dtype=torch.bfloat16, device=dev) if out_bf16 else None
    y_lo = torch.empty((M, N), dtype=torch.bfloat16, device=dev) if (out_bf16 and out_lo) else None
    y_f = torch.empty((M, N), dtype=torch.float32, device=dev) if out_f32 else None
    check(lib.rvae_linear_act_fwd(ctx(dev), xh, xl, wh, wl, _ptr(bias, torch.float32, "bias"), M, N, K, act,
                                  _ptr(y_hi), _ptr(y_lo), _ptr(y_f), _stream()))
    return y_hi, y_lo, y_f


def encode_head_fwd(h, w2, b2, eps, *, want_lo=False, want_z=True, kl_acc=None):
    """mu, logvar (fp32) and z = mu + eps*exp(logvar/2) (bf16 planes) from h [M,K], stacked W2 [2L,K], b2 [2L],
    eps [M,L] (None = 0)."""
    lib = _lib.load()
    hh, hl = _planes(h, "h")
    wh, wl = _planes(w2, "w2")
    ht = h[0] if isinstance(h, (tuple, list)) else h
    wt = w2[0] if isinstance(w2, (tuple, list)) else w2
    M, K = ht.shape
    L = wt.shape[0] // 2
    dev = ht.device
    f = lambda: torch.empty((M, L), dtype=torch.float32, device=dev)
    mu, lv = f(), f()
    z_hi = torch.empty((M, L), dtype=torch.bfloat16, device=dev) if want_z else None
    z_lo = torch.empty_like(z_hi) if (want_z and want_lo) else None
    check(lib.rvae_encode_head_fwd(ctx(dev), hh, hl, wh, wl, _ptr(b2, torch.float32, "b2"), M, L, K,
                                   _ptr(eps, torch.float32, "eps"), _ptr(mu), _ptr(lv), _ptr(z_hi), _ptr(z_lo),
                                   _ptr(kl_acc, torch.float64, "kl_acc"), _stream()))
    return mu, lv, (z_hi, z_lo)


def out_tanh_mse_fwd(h3, w4, b4, x, *, grad_scale: float, tanh_approx=False, want_xhat=True, want_da=True,
                     want_lo=False, mse_acc=None, bias_grad=None):
    lib = _lib.load()
    hh, hl = _planes(h3, "h3")
    wh, wl = _planes(w4, "w4")
    xh, xl = _planes(x, "x")
    ht = h3[0] if isinstance(h3, (tuple, list)) else h3
    wt = w4[0] if isinstance(w4, (tuple, list)) else w4
    M, K = ht.shape
    S = wt.shape[0]
    dev = ht.device
    xhat = torch.empty((M, S), dtype=torch.float32, device=dev) if want_xhat else None
    da_hi = torch.empty((M, S), dtype=torch.bfloat16, device=dev) if want_da else None
    da_lo = torch.empty_like(da_hi) if (want_da and want_lo) else None
    check(lib.rvae_out_tanh_mse_fwd(ctx(dev), hh, hl, wh, wl, _ptr(b4, torch.float32, "b4"), M, S, K, xh, xl,
                                    int(tanh_approx), _ptr(xhat), _ptr(da_hi), _ptr(da_lo), grad_scale,
                                    _ptr(mse_acc, torch.float64, "mse_acc"),
                                    _ptr(bias_grad, torch.float32, "bias_grad"), _stream()))
    return xhat, (da_hi, da_lo)


def dgrad_relu(dy, w, mask, *, want_lo=False, bias_grad=None):
    """dx = (dy @ w) * [mask > 0]; dy [M,Kd], w [Kd,N] (Linear weight, row-major), mask bf16 [M,N] or None."""
    lib = _lib.load()
    dh, dl = _planes(dy, "dy")
    wh, wl = _planes(w, "w")
    dt = dy[0] if isinstance(dy, (tuple, list)) else dy
    wt = w[0] if isinstance(w, (tuple, list)) else w
    M, Kd = dt.shape
    N = wt.shape[1]
    dev = dt.device
    dx_hi = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
    dx_lo = torch.empty_like(dx_hi) if want_lo else None
    check(lib.rvae_dgrad_relu(ctx(dev), dh, dl, wh, wl, M, N, Kd, _ptr(mask, torch.bfloat16, "mask"), _ptr(dx_hi),
                              _ptr(dx_lo), _ptr(bias_grad, torch.float32, "bias_grad"), _stream()))
    return dx_hi, dx_lo


def dgrad_latent(da3, w3, eps, logvar, mu=None, *, g_mu=None, g_logvar=None, kl_grad_scale: float = 0.0,
                 want_lo=False, bias_grad=None):
    """d_ml = [dz + g_mu | dz*eps*exp(logvar/2)/2 + g_logvar] with dz = da3 @ w3; the additive terms are the KL
    gradient computed from (mu, logvar, kl_grad_scale) unless external g_mu / g_logvar are given."""
    lib = _lib.load()
    dh, dl = _planes(da3, "da3")
    wh, wl = _planes(w3, "w3")
    dt = da3[0] if isinstance(da3, (tuple, list)) else da3
    wt = w3[0] if isinstance(w3, (tuple, list)) else w3
    M, H = dt.shape
    L = wt.shape[1]
    dev = dt.device
    hi = torch.empty((M, 2 * L), dtype=torch.bfloat16, device=dev)
    lo = torch.empty_like(hi) if want_lo else None
    dz = torch.empty((M, L), dtype=torch.float32, device=dev)
    check(lib.rvae_dgrad_latent(ctx(dev), dh, dl, wh, wl, M, L, H, _ptr(eps, torch.float32, "eps"),
                                _ptr(logvar, torch.float32, "logvar"), _ptr(mu, torch.float32, "mu"),
                                _ptr(g_mu, torch.float32, "g_mu"), _ptr(g_logvar, torch.float32, "g_logvar"),
                                kl_grad_scale, _ptr(dz), _ptr(hi), _ptr(lo),
                                _ptr(bias_grad, torch.float32, "bias_grad"), _stream()))
    return hi, lo


def wgrad(dy, x, *, out: Optional[torch.Tensor] = None, k_splits: int = 0) -> torch.Tensor:
    """dW = dy.T @ x; dy [B,M], x [B,N] -> fp32 [M,N]."""
    lib = _lib.load()
    dh, dl = _planes(dy, "dy")
    xh, xl = _planes(x, "x")
    dt = dy[0] if isinstance(dy, (tuple, list)) else dy
    xt = x[0] if isinstance(x, (tuple, list)) else x
    B, M = dt.shape
    N = xt.shape[1]
    if out is None:
        out = torch.zeros((M, N), dtype=torch.float32, device=dt.device)
    check(lib.rvae_wgrad(ctx(dt.device), dh, dl, xh, xl, B, M, N, _ptr(out, torch.float32, "out"), 1, k_splits,
                         _stream()))
    return out
