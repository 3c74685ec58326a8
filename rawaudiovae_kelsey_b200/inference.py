"""Inference API for the reference's tutorial pattern (tutorial.ipynb, SURVEY.md 3.4 / 8f N3):

    encode_audio(model, wav)                      raw_to_z_dist        tutorial.ipynb:456-470 (cells 13-14)
    lerp_latents(mu_a, lv_a, mu_b, lv_b, alpha)   latent interpolation tutorial.ipynb:496-510 (global alpha),
                                                                       :905-932 (per-frame float64 alpha from interp1d)
    decode_latents(model, z)                      raw_model.decode     tutorial.ipynb:506,923
    resynthesize(frames, mode, hop)               frames.view(-1)      tutorial.ipynb:543,932,1289 ('concat');
                                                  overlap-add of hop-strided frames ('ola', new - SURVEY.md Q8)
    interpolate(model, ...)                       the whole chain lerp -> reparameterize -> decode as ONE enqueue per
                                                  batch: z is written straight into fc3's bf16 operand
    evaluate_audio(model, wav, kl_beta)           per-frame loss_function terms of held-out audio (rawvae/model.py:
                                                  38-46 on the test_dataset of train.py:153-155) and their mean

The audio lives in HBM once; frames are gathered by index into fc1's operand (never materialised in fp32); latents
of all frames are written into one preallocated tensor (no per-batch torch.cat). CUDA only - CPU tensors raise.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib, ops
from .model import VAE, FrameBatch


def _device_of(model: VAE) -> torch.device:
    p = model.fc1.weight
    if not p.is_cuda:
        raise _lib.RvaeError("the model is on the CPU: call model.to('cuda') - there is no CPU fallback")
    return p.device


def _audio_to_device(wav, dev: torch.device, multiple: int) -> torch.Tensor:
    """1-D float32 / int16 samples in HBM, zero-padded on the right to a multiple of `multiple` (the reference's
    datasets pad the same way: rawvae/dataset.py:102-104 to a multiple of hop, :141-143 to a multiple of S)."""
    if isinstance(wav, np.ndarray):
        wav = torch.from_numpy(np.ascontiguousarray(wav))
    if not isinstance(wav, torch.Tensor) or wav.dim() != 1:
        raise TypeError("wav must be a 1-D numpy array or torch tensor of samples")
    if wav.dtype not in (torch.float32, torch.int16):
        wav = wav.to(torch.float32)
    wav = wav.to(dev)
    pad = (-wav.numel()) % multiple
    if pad:
        wav = torch.nn.functional.pad(wav, (0, pad))
    return wav.contiguous()


def frame_count(n_samples: int, segment_length: int, hop: Optional[int] = None) -> int:
    """Frames the reference's datasets produce: TestDataset (hop None: non-overlapping, rawvae/dataset.py:160) or
    AudioDataset (rawvae/dataset.py:121)."""
    if hop is None:
        return -(-n_samples // segment_length)
    padded = -(-n_samples // hop) * hop
    return padded // hop - segment_length // hop + 1


@torch.no_grad()
def encode_audio(model: VAE, wav, *, hop: Optional[int] = None, batch_size: int = 16384
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
    """(mu, logvar), fp32 [n_frames, L], of every frame of `wav`: TestDataset framing by default (hop = S, the
    notebook's cells 13-14), AudioDataset framing when `hop` is given (its "extensions" cells)."""
    dev = _device_of(model)
    S, L = model.segment_length, model.latent_dim
    step = S if hop is None else int(hop)
    if S % step != 0:
        raise ValueError("segment_length {} is not a multiple of hop_size {}".format(S, step))
    n = int(wav.shape[0])
    audio = _audio_to_device(wav, dev, step)
    N = frame_count(n, S, hop)
    mu = torch.empty((N, L), dtype=torch.float32, device=dev)
    lv = torch.empty_like(mu)
    for lo in range(0, N, batch_size):
        hi = min(N, lo + batch_size)
        plan = model._load(FrameBatch(audio, hi - lo, step, S, first_frame=lo))
        plan.set_outputs(mu[lo:hi], lv[lo:hi], None)     # row slices of the result: no per-batch cat
        plan.encode()
        plan.set_outputs(None, None, None)
    return mu, lv


def _alpha_tensor(alpha, n: int, dev: torch.device) -> torch.Tensor:
    if isinstance(alpha, (int, float)):
        return torch.full((n,), float(alpha), dtype=torch.float64, device=dev)
    if isinstance(alpha, np.ndarray):
        alpha = torch.from_numpy(alpha)
    alpha = alpha.to(dev)
    if alpha.dtype not in (torch.float32, torch.float64):
        alpha = alpha.to(torch.float64)
    if alpha.dim() == 2 and alpha.shape[1] >= 1:   # the notebook repeats alpha over the latent dimension (cell 37)
        alpha = alpha[:, 0]
    if alpha.numel() != n:
        raise ValueError(f"alpha has {alpha.numel()} entries, expected one per frame ({n})")
    return alpha.reshape(n).contiguous()


def _noise(model: VAE, shape, dev) -> torch.Tensor:
    if model.eps_source == "torch":
        return torch.randn(shape, device=dev)
    seed, off = model._eps_args()
    return ops.randn(shape, seed, off, device=dev)


@torch.no_grad()
def lerp_latents(mu_a, lv_a, mu_b, lv_b, alpha, eps: Optional[torch.Tensor] = None, *, sample: bool = True,
                 return_dist: bool = False, seed: Optional[int] = None):
    """z = mu + eps * exp(logvar / 2) with mu = (1 - alpha) mu_a + alpha mu_b, logvar likewise; alpha is a scalar or
    one value per frame (float64 accepted, as interp1d returns it). eps None draws Philox noise (reparameterize keeps
    sampling at inference, as the reference's does); sample=False gives the mean path (eps = 0).
    Returns z, or (z, mu, logvar) with return_dist=True."""
    if not mu_a.is_cuda:
        raise _lib.RvaeError("lerp_latents: CPU tensors are not supported (no CPU fallback)")
    n, L = mu_a.shape
    dev = mu_a.device
    c = lambda t: t.to(torch.float32).contiguous()
    al = _alpha_tensor(alpha, n, dev)
    if eps is None and sample:
        eps = ops.randn((n, L), seed if seed is not None else torch.initial_seed() & 0x7FFFFFFFFFFFFFFF, 0, device=dev)
    z, mu, lv = ops.lerp_reparameterize(c(mu_a), c(lv_a), c(mu_b), c(lv_b), al, None if eps is None else c(eps),
                                        want_z=True, want_dist=return_dist)
    return (z, mu, lv) if return_dist else z


@torch.no_grad()
def decode_latents(model: VAE, z: torch.Tensor, *, batch_size: int = 16384) -> torch.Tensor:
    """frames = tanh(fc4(relu(fc3 z))), fp32 [n, S] (rawvae/model.py:28-30), batch by batch into one tensor."""
    dev = _device_of(model)
    z = z.reshape(-1, model.latent_dim).to(device=dev, dtype=torch.float32).contiguous()
    n = z.shape[0]
    out = torch.empty((n, model.segment_length), dtype=torch.float32, device=dev)
    for lo in range(0, n, batch_size):
        hi = min(n, lo + batch_size)
        model._plan_for(hi - lo).decode(z[lo:hi], out[lo:hi])
    return out


@torch.no_grad()
def interpolate(model: VAE, mu_a, lv_a, mu_b, lv_b, alpha: Union[float, Sequence[float], torch.Tensor, np.ndarray],
                eps: Optional[torch.Tensor] = None, *, sample: bool = True, batch_size: int = 16384) -> torch.Tensor:
    """Latent interpolation -> reparameterize -> decode as one chained enqueue per batch (rvae_plan_decode_lerp): the
    interpolated z never exists in fp32 in HBM. alpha: a tensor / array with one value per frame (cell 37), or a
    list of global values (cell 16: `for interpolation in interpolation_range`, results concatenated along dim 0)."""
    dev = _device_of(model)
    n, L = mu_a.shape
    S = model.segment_length
    c = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()
    mu_a, lv_a, mu_b, lv_b = c(mu_a), c(lv_a), c(mu_b), c(lv_b)
    sweep = isinstance(alpha, (list, tuple))
    alphas = [_alpha_tensor(a, n, dev) for a in alpha] if sweep else [_alpha_tensor(alpha, n, dev)]
    out = torch.empty((len(alphas) * n, S), dtype=torch.float32, device=dev)
    for k, al in enumerate(alphas):
        e = eps
        if e is None and sample:
            e = _noise(model, (n, L), dev)        # fresh noise per interpolation value, as reparameterize draws it
        e = None if e is None else c(e)
        for lo in range(0, n, batch_size):
            hi = min(n, lo + batch_size)
            plan = model._plan_for(hi - lo)
            plan.decode_lerp(mu_a[lo:hi], lv_a[lo:hi], mu_b[lo:hi], lv_b[lo:hi], al[lo:hi],
                             None if e is None else e[lo:hi], out[k * n + lo:k * n + hi])
    return out


@torch.no_grad()
def resynthesize(frames: torch.Tensor, mode: str = "concat", hop: Optional[int] = None,
                 n_out: Optional[int] = None) -> torch.Tensor:
    """Frames -> audio. 'concat': frames.view(-1), what the reference does everywhere (train_iterable.py:246,
    tutorial.ipynb:543,932,1289; exact for TestDataset framing, an S/hop-times time-stretch for hop-strided frames -
    the notebook's "hacky.wav"). 'ola': overlap-add of frames at stride `hop`, normalised by the per-sample overlap
    count, so that ola(AudioDataset frames of x) == padded x (new op; SURVEY.md Q8: unpinned by the reference)."""
    if not frames.is_cuda:
        raise _lib.RvaeError("resynthesize: CPU tensors are not supported (no CPU fallback)")
    frames = frames.to(torch.float32).contiguous()
    if mode == "concat":
        return frames.reshape(-1)
    if mode != "ola":
        raise ValueError("mode must be 'concat' or 'ola'")
    if hop is None:
        raise ValueError("mode='ola' needs the hop the frames were cut with")
    return ops.overlap_add(frames, int(hop), n_out)


@dataclass
class Evaluation:
    """evaluate_audio's result. reconstruction / kl: fp32 [n_frames], the per-frame terms of loss_function;
    loss = mean(reconstruction + kl_beta * kl), reconstruction_mean = mean(reconstruction), kl_mean = mean(kl), each
    summed in float64."""
    reconstruction: torch.Tensor
    kl: torch.Tensor
    loss: float
    reconstruction_mean: float
    kl_mean: float


@torch.no_grad()
def evaluate_audio(model: VAE, wav, kl_beta: float, *, hop: Optional[int] = None, batch_size: int = 16384,
                   sample: bool = True, seed: int = 0) -> Evaluation:
    """Score held-out audio: per frame, the reconstruction error and KL divergence of loss_function
    (rawvae/model.py:38-46), and their dataset mean - the number the reference's test_dataset never produces
    (train.py:153-155, train_iterable.py:170-172 load it for listening only).

    Framing as encode_audio: TestDataset by default, AudioDataset at stride `hop` when given. Per batch: the frames are
    loaded into the model's plan, run through a plain forward and scored by rvae_frame_loss against the exact audio
    samples (x is never rounded to bf16). Noise: sample=True draws eps from Philox(seed, offset 0) keyed by frame
    index, so results do not depend on batch_size and evaluations of different checkpoints share their noise;
    sample=False is the mean path (eps = 0). The model's noise counter, parameters, gradients, optimizer state and a
    batch a FusedTrainStep has prefetched are left as they were."""
    dev = _device_of(model)
    S, L = model.segment_length, model.latent_dim
    step = S if hop is None else int(hop)
    if S % step != 0:
        raise ValueError("segment_length {} is not a multiple of hop_size {}".format(S, step))
    if batch_size <= 0:
        raise ValueError("batch_size must be positive")
    n = int(wav.shape[0])
    audio = _audio_to_device(wav, dev, step)
    N = frame_count(n, S, hop)
    if N <= 0:
        raise ValueError("{} samples give no frame of {} samples".format(n, S))
    rec = torch.empty(N, dtype=torch.float32, device=dev)
    kl = torch.empty_like(rec)
    zero = None if sample else torch.zeros((min(batch_size, N), L), dtype=torch.float32, device=dev)
    for lo in range(0, N, batch_size):
        hi = min(N, lo + batch_size)
        b = hi - lo
        plan = model._load(FrameBatch(audio, b, step, S, first_frame=lo))
        plan.set_eps(ops.randn((b, L), int(seed) & 0xFFFFFFFFFFFFFFFF, 0, device=dev, elem_base=lo * L) if sample
                     else zero[:b])
        plan.forward(0.0, fused_loss=False, want_xhat=True)
        ops.frame_loss(plan.xhat(), plan.latent("mu"), plan.latent("logvar"), audio, lo, step, rec[lo:hi], kl[lo:hi])
    r64, k64 = rec.double(), kl.double()
    sums = torch.stack([(r64 + float(kl_beta) * k64).sum(), r64.sum(), k64.sum()]).cpu().tolist()
    return Evaluation(rec, kl, sums[0] / N, sums[1] / N, sums[2] / N)


@torch.no_grad()
def reconstruct_audio(model: VAE, wav, *, hop: Optional[int] = None, mode: Optional[str] = None,
                      batch_size: int = 16384, sample: bool = True, eps: Optional[torch.Tensor] = None) -> torch.Tensor:
    """wav -> frames -> encode -> reparameterize -> decode -> audio, streamed batch by batch (BASELINE.json configs[4]:
    the widened-VAE inference pattern; also the trainers' test-audio reconstruction, train_iterable.py:228-246).

    hop None: TestDataset framing (non-overlapping frames) + concatenation, as the reference resynthesises.
    hop given: AudioDataset framing at stride hop; mode 'ola' (default) overlap-adds across batch boundaries - the
    last S/hop - 1 decoded frames of a batch are carried into the next one, each output sample is finalised once -
    so memory stays O(batch) however long the audio is; mode 'concat' reproduces the notebook's frames.view(-1).
    The wav stays in HBM as it came (int16 or float32); frames are never materialised in fp32; decoded frames live
    in one [S/hop - 1 + batch, S] buffer. Noise: `eps` [n_frames, L] if given, else Philox per frame (sample=True)
    or none (sample=False: the mean path)."""
    dev = _device_of(model)
    S, L = model.segment_length, model.latent_dim
    step = S if hop is None else int(hop)
    if S % step != 0:
        raise ValueError("segment_length {} is not a multiple of hop_size {}".format(S, step))
    n = int(wav.shape[0])
    audio = _audio_to_device(wav, dev, step)
    N = frame_count(n, S, hop)
    ola = hop is not None and (mode or "ola") == "ola"
    if hop is not None and (mode or "ola") not in ("ola", "concat"):
        raise ValueError("mode must be 'concat' or 'ola'")
    r = S // step if ola else 1                         # frames covering one sample
    n_out = (N - 1) * step + S if ola else N * S
    out = torch.empty(n_out, dtype=torch.float32, device=dev)
    B = min(batch_size, N)
    buf = torch.empty((r - 1 + B, S), dtype=torch.float32, device=dev)   # [carry of the previous batch | this batch]
    mu = torch.empty((B, L), dtype=torch.float32, device=dev)
    lv = torch.empty_like(mu)
    zero = torch.zeros(B, dtype=torch.float32, device=dev)
    seed, off = model._eps_args() if (eps is None and sample and model.eps_source != "torch") else (0, 0)
    for lo in range(0, N, B):
        hi = min(N, lo + B)
        b = hi - lo
        plan = model._load(FrameBatch(audio, b, step, S, first_frame=lo))
        plan.set_outputs(mu[:b], lv[:b], None)
        plan.encode()
        plan.set_outputs(None, None, None)
        if eps is not None:
            e = eps[lo:hi].to(device=dev, dtype=torch.float32).contiguous()
        elif not sample:
            e = None
        elif model.eps_source == "torch":
            e = torch.randn((b, L), device=dev)
        else:
            e = ops.randn((b, L), seed, off, device=dev, elem_base=lo * L)    # one noise tensor over all frames
        frames = buf[r - 1:r - 1 + b]
        plan.decode_lerp(mu[:b], lv[:b], mu[:b], lv[:b], zero[:b], e, frames)  # alpha = 0: z goes straight to fc3
        if not ola:
            out[lo * S:hi * S].copy_(frames.reshape(-1))
            continue
        # finalise samples [lo * hop, hi * hop) (+ the tail after the last frame): every frame covering them is in buf
        valid = min(r - 1, lo)                       # carried frames that exist (fewer than r - 1 near the start)
        src = buf[r - 1 - valid:r - 1 + b]
        t0 = valid * step                            # local sample index of global sample lo * hop
        cnt = (b * step) if hi < N else (b - 1) * step + S
        ops.overlap_add(src, step, cnt, t_begin=t0, out=out[lo * step:lo * step + cnt])
        if hi < N and r > 1:
            buf[:r - 1].copy_(buf[b:b + r - 1].clone())     # carry the last r - 1 frames (b >= r - 1 for full batches)
    return out
