"""The exponential moving average of the weights without a GPU: decay validation in ExponentialMovingAverage and the
step constructors, the trainers' ini key, the argument checks of the C entries, and the fp64 reference of the EMA
recurrence against torch's AveragedModel on CPU tensors."""
import configparser
import math
from pathlib import Path

import numpy as np
import pytest
import torch
from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn

from rawaudiovae_kelsey_b200 import _lib

ROOT = Path(__file__).resolve().parents[1]
BAD = [-0.1, 1.0000001, 2, math.inf, -math.inf, math.nan, "0.9", True, None, [0.9], torch.tensor(0.9)]


@pytest.mark.parametrize("bad", BAD, ids=[repr(b) for b in BAD])
def test_decay_validation(bad):
    from rawaudiovae_kelsey_b200.ema import ExponentialMovingAverage, check_ema_decay
    with pytest.raises(ValueError, match="decay"):
        check_ema_decay(bad)
    with pytest.raises(ValueError, match="decay"):
        ExponentialMovingAverage(None, decay=bad)        # raised before the model (or a GPU) is touched


def test_decay_accepts_the_closed_interval():
    from rawaudiovae_kelsey_b200.ema import check_ema_decay
    for v in (0, 0.0, 0.5, 0.999, 1, 1.0):
        assert check_ema_decay(v) == float(v)


@pytest.mark.parametrize("cls", ["fused", "dp"])
def test_step_constructors_check_the_ema(cls):
    from rawaudiovae_kelsey_b200.dist import DataParallelTrainStep
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    make = FusedTrainStep if cls == "fused" else DataParallelTrainStep
    assert make(None, None, 0.5).ema is None
    for bad in (0.999, "ema", object()):
        with pytest.raises(ValueError, match="ema"):
            make(None, None, 0.5, ema=bad)


def _cfg(path, **training):
    cfg = configparser.ConfigParser()
    cfg.read(ROOT / path)
    for k, v in training.items():
        cfg["training"][k] = str(v)
    return cfg


@pytest.mark.parametrize("path", ["default.ini", "kelsey_iterable.ini"])
def test_ini_key(path):
    from rawaudiovae_kelsey_b200.trainer import _ema_decay
    assert "# ema_decay = 0.999" in (ROOT / path).read_text()
    assert _ema_decay(_cfg(path)) is None
    assert _ema_decay(_cfg(path, ema_decay="")) is None
    assert _ema_decay(_cfg(path, ema_decay="0.999")) == 0.999
    assert _ema_decay(_cfg(path, ema_decay="0")) == 0.0
    assert _ema_decay(_cfg(path, ema_decay="1")) == 1.0
    for bad in ("-0.1", "1.5", "nan", "inf", "one", "0.9.9"):
        with pytest.raises(ValueError, match="ema_decay"):
            _ema_decay(_cfg(path, ema_decay=bad))


def test_device_record_holds_the_decay_after_the_threshold():
    import ctypes as C
    import struct
    from rawaudiovae_kelsey_b200.schedule import DeviceRecord
    rec = DeviceRecord.__new__(DeviceRecord)      # the layout only: no device tensor
    rec.tensor = torch.zeros(C.sizeof(_lib.Hparams) + 16, dtype=torch.uint8)
    assert rec.ema_decay_ptr - rec.max_norm_ptr == 8
    assert rec.ema_decay_ptr + 8 == rec.tensor.data_ptr() + rec.tensor.numel()
    assert struct.calcsize("<dd") == 16


def test_entries_are_declared_and_check_arguments_before_the_plan():
    lib = _lib.load()
    assert "rvae_plan_set_ema" in _lib.SIGNATURES and "rvae_ema_update" in _lib.SIGNATURES
    hdr = (ROOT / "include" / "rvae_b200.h").read_text()
    assert "int rvae_plan_set_ema(rvae_plan* plan, float* ema, const double* decay_dev, int64_t* count_dev);" in hdr
    assert ("int rvae_ema_update(rvae_ctx* ctx, float* ema, const float* params, int64_t n, const double* decay_dev,\n"
            "                    int64_t* count_dev, void* stream);") in hdr
    # refused before the (bogus) plan pointer is read
    assert lib.rvae_plan_set_ema(8, 16, None, 16) == 1
    assert b"decay" in lib.rvae_last_error()
    assert lib.rvae_plan_set_ema(8, 16, 16, None) == 1
    assert lib.rvae_plan_set_ema(8, 20, 16, 16) == 1
    assert b"aligned" in lib.rvae_last_error()
    assert lib.rvae_plan_set_ema(None, 16, 16, 16) == 1
    assert lib.rvae_plan_set_ema(None, None, None, None) == 1       # off, but there is no plan
    # rvae_ema_update: null buffers and n < 0 before the ctx is used
    assert lib.rvae_ema_update(8, None, 16, 4, 16, 16, None) == 1
    assert lib.rvae_ema_update(8, 16, 16, -1, 16, 16, None) == 1
    assert lib.rvae_ema_update(8, 16, 16, 4, None, 16, None) == 1
    assert lib.rvae_ema_update(8, 16, 16, 4, 16, None, None) == 1
    assert lib.rvae_ema_update(None, 16, 16, 4, 16, 16, None) == 1
    assert b"rvae_ctx" in lib.rvae_last_error()
    assert lib.rvae_abi_version() == 5


def ema_reference(snapshots, decay):
    """fp64 host reference of the recurrence: e = p_0, then e = e + (1 - decay) (p_k - e)."""
    w = 1.0 - decay
    e = snapshots[0].double().clone()
    for p in snapshots[1:]:
        e = e + w * (p.double() - e)
    return e


def lerp32(e, p, w):
    """torch's two-branch lerp in fp32 (numpy, no contraction): the formula the kernels evaluate."""
    e, p, w = np.float32(e), np.float32(p), np.float32(w)
    return e + w * (p - e) if abs(w) < 0.5 else p - (p - e) * (np.float32(1) - w)


@pytest.mark.parametrize("decay", [0.0, 0.5, 0.9, 0.999, 1.0])
def test_reference_agrees_with_averaged_model(decay):
    gen = torch.Generator().manual_seed(0)
    lin = torch.nn.Linear(16, 8)
    avg = AveragedModel(lin, multi_avg_fn=get_ema_multi_avg_fn(decay))
    snaps = []
    for _ in range(12):
        with torch.no_grad():
            lin.weight.copy_(torch.randn(8, 16, generator=gen))
        avg.update_parameters(lin)
        snaps.append(lin.weight.detach().clone())
    assert int(avg.n_averaged) == 12
    ref = ema_reference(snaps, decay)
    got = avg.module.weight.detach().double()
    assert torch.allclose(got, ref, rtol=0, atol=1e-5), float((got - ref).abs().max())
    # the weight torch uses: 1 - decay formed in double and rounded to fp32 once
    w = np.float32(1.0 - decay)
    e = snaps[0].numpy().astype(np.float32)
    for p in snaps[1:]:
        e = np.vectorize(lerp32, otypes=[np.float32])(e, p.numpy(), w)
    assert np.allclose(e, got.numpy(), rtol=0, atol=2e-6)


def test_first_update_copies_and_non_finite_values_propagate():
    lin = torch.nn.Linear(2, 1, bias=False)
    avg = AveragedModel(lin, multi_avg_fn=get_ema_multi_avg_fn(0.9))
    with torch.no_grad():
        lin.weight.copy_(torch.tensor([[1.0, 2.0]]))
    avg.update_parameters(lin)
    assert torch.equal(avg.module.weight, lin.weight)
    with torch.no_grad():
        lin.weight.copy_(torch.tensor([[math.inf, math.nan]]))
    avg.update_parameters(lin)
    w = avg.module.weight.detach()[0]
    assert math.isinf(float(w[0])) and math.isnan(float(w[1]))
    assert math.isinf(lerp32(1.0, math.inf, np.float32(0.1))) and math.isnan(lerp32(2.0, math.nan, np.float32(0.1)))
