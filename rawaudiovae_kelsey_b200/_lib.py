"""ctypes binding of librvae_b200.so (include/rvae_b200.h).

There is no fallback: if the CUDA extension is missing or fails to load, every entry point raises. The oracle
under oracle/ is test infrastructure and is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import threading
from pathlib import Path

from . import _build

_LIB = None
_LOCK = threading.Lock()
ABI_VERSION = 5

c_void_p, c_int, c_int64, c_uint64, c_float, c_size_t = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_float, C.c_size_t
c_double = C.c_double


class RvaeError(RuntimeError):
    """A non-zero return code from librvae_b200 (message from rvae_last_error())."""


class Layout(C.Structure):
    _fields_ = [(n, c_int64) for n in ("w1", "w2", "w3", "w4", "b1", "b2", "b3", "b4", "total")]


class PlanBuffers(C.Structure):
    _fields_ = [(n, c_void_p) for n in
                ("params", "grads", "exp_avg", "exp_avg_sq", "step", "shadow_hi", "shadow_lo", "workspace")]


class Hparams(C.Structure):
    """rvae_hparams: the device-resident hyper-parameter record of a scheduled training step (112 bytes)."""
    _fields_ = [(n, c_double) for n in ("lr", "beta1", "beta2", "eps", "weight_decay", "kl_beta", "lr_min",
                                        "kl_beta_start", "kl_cycle_ratio")] + \
               [(n, c_int64) for n in ("total_steps", "warmup_steps", "kl_anneal_steps", "kl_cycles")] + \
               [(n, C.c_int32) for n in ("lr_schedule", "kl_anneal")]


# name -> (restype, argtypes); every symbol declared in include/rvae_b200.h
P = c_void_p
SIGNATURES = {
    "rvae_abi_version": (c_int, []),
    "rvae_build_experiments": (c_int, []),
    "rvae_last_error": (C.c_char_p, []),
    "rvae_ctx_create": (c_int, [c_int, C.POINTER(P)]),
    "rvae_ctx_destroy": (None, [P]),
    "rvae_ctx_num_sms": (c_int, [P]),
    "rvae_ctx_launch_count": (c_uint64, [P]),
    "rvae_dp_unique_id": (c_int, [P, C.c_char_p, P]),
    "rvae_dp_init": (c_int, [P, C.c_char_p, P, c_int, c_int]),
    "rvae_dp_world": (c_int, [P]),
    "rvae_dp_sym_alloc": (c_int, [P, c_size_t, C.POINTER(P), P]),
    "rvae_dp_sym_open": (c_int, [P, P, c_int, c_int]),
    "rvae_dp_sym_flag_bytes": (c_size_t, []),
    "rvae_dp_sym_adopt": (c_int, [P, C.POINTER(P), P, c_size_t, c_int, c_int]),
    "rvae_dp_uses_multicast": (c_int, [P]),
    "rvae_dp_allreduce": (c_int, [P, P, c_int64, c_int, P]),
    "rvae_frame_gather": (c_int, [P, P, c_int, c_int64, P, c_int64, c_int64, c_int, c_int, P, P, P, P]),
    "rvae_overlap_add": (c_int, [P, P, c_int64, c_int, c_int, P, c_int64, c_int64, P]),
    "rvae_randn": (c_int, [P, P, c_int64, c_uint64, c_uint64, c_int64, P]),
    "rvae_lerp_reparameterize": (c_int, [P, P, P, P, P, P, c_int, P, c_int64, c_int, P, P, P, P]),
    "rvae_dp_status": (c_int, [P, C.POINTER(C.c_uint)]),
    "rvae_plan_set_noise_rows": (c_int, [P, c_int64]),
    "rvae_plan_decode_lerp": (c_int, [P, P, P, P, P, P, c_int, P, c_int, P, P]),
    "rvae_split_bf16": (c_int, [P, P, c_int64, P, P, P]),
    "rvae_reparameterize": (c_int, [P, P, P, P, c_int64, P, P]),
    "rvae_loss_fwd": (c_int, [P, P, P, P, P, c_int64, c_int, c_int, c_float, P, P, P]),
    "rvae_frame_loss": (c_int, [P, P, c_int, P, P, c_int, c_int64, c_int, c_int, P, c_int, c_int64, c_int64, c_int, P,
                                P, P]),
    "rvae_loss_bwd": (c_int, [P, P, P, P, P, c_int64, c_int, c_int, c_float, P, P, P, P, P]),
    "rvae_tanh_bwd": (c_int, [P, P, P, c_int64, P, P, P]),
    "rvae_colsum": (c_int, [P, P, P, c_int64, c_int, c_int, P, c_int, P]),
    "rvae_step_inc": (c_int, [P, P, P]),
    "rvae_adam_step": (c_int, [P, P, P, P, P, c_int64, c_double, c_double, c_double, c_double, c_double, c_float, P, P,
                               P, P]),
    "rvae_param_histogram_bytes": (c_size_t, [c_int, c_int]),
    "rvae_param_histogram": (c_int, [P, P, P, P, c_int, P, c_int, P, P]),
    "rvae_param_histogram_rows": (c_int, [P, P, P, P, P, P, c_int, P, c_int, P, P]),
    "rvae_linear_act_fwd": (c_int, [P, P, P, P, P, P, c_int, c_int, c_int, c_int, P, P, P, P]),
    "rvae_encode_head_fwd": (c_int, [P, P, P, P, P, P, c_int, c_int, c_int, P, P, P, P, P, P, P]),
    "rvae_out_tanh_mse_fwd": (c_int, [P, P, P, P, P, P, c_int, c_int, c_int, P, P, c_int, P, P, P, c_float, P, P, P]),
    "rvae_dgrad_relu": (c_int, [P, P, P, P, P, c_int, c_int, c_int, P, P, P, P, P]),
    "rvae_dgrad_latent": (c_int, [P, P, P, P, P, c_int, c_int, c_int, P, P, P, P, P, c_float, P, P, P, P, P]),
    "rvae_wgrad": (c_int, [P, P, P, P, P, c_int, c_int, c_int, P, c_int, c_int, P]),
    "rvae_param_layout": (c_int, [c_int, c_int, c_int, C.POINTER(Layout)]),
    "rvae_param_layout_padded": (c_int, [c_int, c_int, c_int, C.POINTER(Layout), C.POINTER(c_int), C.POINTER(c_int),
                                         C.POINTER(c_int)]),
    "rvae_plan_create": (c_int, [P, c_int, c_int, c_int, c_int, c_int, C.POINTER(P)]),
    "rvae_plan_destroy": (None, [P]),
    "rvae_plan_workspace_bytes": (c_size_t, [P]),
    "rvae_plan_bind": (c_int, [P, C.POINTER(PlanBuffers)]),
    "rvae_plan_sync_shadow": (c_int, [P, P]),
    "rvae_plan_load_frames": (c_int, [P, P, c_int, c_int64, P, c_int64, c_int, c_int, c_int, P]),
    "rvae_plan_load_batch": (c_int, [P, P, c_int, P]),
    "rvae_plan_set_eps": (c_int, [P, P, P]),
    "rvae_plan_gen_eps": (c_int, [P, c_uint64, c_uint64, c_int, P]),
    "rvae_plan_set_outputs": (c_int, [P, P, P, P]),
    "rvae_plan_enable_dp": (c_int, [P, c_int]),
    "rvae_plan_set_global_batch": (c_int, [P, c_int64]),
    "rvae_plan_forward": (c_int, [P, c_float, c_int, c_int, P]),
    "rvae_plan_backward": (c_int, [P, c_int, P]),
    "rvae_plan_backward_external": (c_int, [P, P, P, P, P, P, P]),
    "rvae_plan_finish_loss": (c_int, [P, c_float, P, c_int, P]),
    "rvae_plan_finish_loss_deferred": (c_int, [P, c_float, P, c_int]),
    "rvae_plan_prefetch_frames": (c_int, [P, P, c_int, c_int64, P, c_int64, c_int, c_int, c_uint64, c_uint64, c_int]),
    "rvae_plan_swap_prefetched": (c_int, [P]),
    "rvae_plan_prefetched_batch": (c_int, [P]),
    "rvae_plan_note_prefetched": (c_int, [P, c_int, c_int]),
    "rvae_plan_span_supported": (c_int, [P, c_int, c_int]),
    "rvae_plan_load_span": (c_int, [P, P, c_int, c_int64, P, c_int64, c_int, c_int, P]),
    "rvae_plan_prefetch_span": (c_int, [P, P, c_int, c_int64, P, c_int64, c_int, c_int, c_uint64, c_uint64, c_int]),
    "rvae_plan_join_background": (c_int, [P, P]),
    "rvae_plan_adam_buckets": (c_int, [P, C.c_uint, c_double, c_double, c_double, c_double, c_double, c_float, c_int, P]),
    "rvae_plan_adam": (c_int, [P, c_double, c_double, c_double, c_double, c_double, c_float, c_int, P]),
    "rvae_plan_train_step": (c_int, [P, c_float, c_double, c_double, c_double, c_double, c_double, c_int, P, c_int, P]),
    "rvae_plan_train_step_hp": (c_int, [P, P, c_int, P, c_int, P]),
    "rvae_plan_set_grad_clip": (c_int, [P, P, P, c_int]),
    "rvae_plan_grad_norm": (c_int, [P, P, P]),
    "rvae_hparams_check": (c_int, [C.POINTER(Hparams)]),
    "rvae_hparams_eval": (c_int, [P, P, P, c_int, P, P, P]),
    "rvae_plan_mu": (P, [P]),
    "rvae_plan_logvar": (P, [P]),
    "rvae_plan_xhat": (P, [P]),
    "rvae_plan_eps": (P, [P]),
    "rvae_plan_activation": (c_int, [P, c_int, C.POINTER(P), C.POINTER(P), C.POINTER(c_int)]),
    "rvae_plan_bucket": (c_int, [P, c_int, C.POINTER(P), C.POINTER(c_int64)]),
    "rvae_plan_enable_timing": (c_int, [P, c_int]),
    "rvae_plan_read_timing": (c_int, [P, P, P, P]),
    "rvae_debug_set_trace": (c_int, [P, P, c_int]),
    "rvae_debug_set_aux_trace": (c_int, [P, P, c_int]),
    "rvae_plan_decode": (c_int, [P, P, c_int, P, P]),
    "rvae_plan_encode": (c_int, [P, P]),
}


def library_path() -> Path:
    return _build.LIB_PATH


def _stale() -> bool:
    """The library exists but was built from other sources (fingerprint mismatch) and can be rebuilt here. Where the
    sources or nvcc are unavailable (a deployed copy), the existing library is used as it is."""
    try:
        return _build.needs_build() and bool(_build._nvcc())
    except Exception:
        return False


def load(build_if_missing: bool = True):
    """Load librvae_b200.so (building it in-tree with nvcc if it is absent). Raises if that is impossible."""
    global _LIB
    if _LIB is not None:
        return _LIB
    with _LOCK:
        if _LIB is not None:
            return _LIB
        path = library_path()
        stale = path.exists() and _stale()
        if not path.exists() or stale:
            if not build_if_missing:
                raise RvaeError(f"{path} is {'stale' if stale else 'missing'}: the CUDA extension has not been built "
                                "(no CPU fallback exists)")
            _build.build()
        lib = C.CDLL(str(path))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        got = lib.rvae_abi_version()
        if got != ABI_VERSION:
            raise RvaeError(f"librvae_b200 ABI version {got}, expected {ABI_VERSION}")
        _LIB = lib
    return _LIB


def check(rc: int) -> None:
    if rc != 0:
        msg = load().rvae_last_error()
        raise RvaeError(f"librvae_b200 error {rc}: {msg.decode() if msg else '?'}")
