"""Gradient-norm clipping without a GPU: max_grad_norm validation in the step constructors, the trainers' ini key, the
fp64 clipping reference the GPU tests use against torch.nn.utils.clip_grad_norm_, and the argument checks of the C
entries."""
import configparser
import math
from pathlib import Path

import pytest
import torch

from rawaudiovae_kelsey_b200 import _lib

ROOT = Path(__file__).resolve().parents[1]
BAD = [0, 0.0, -1.0, -math.inf, math.nan, "1.0", True, [1.0], torch.tensor(1.0)]


def clip_grad_norm(grads, max_norm):
    """fp64 reference of a clipping step: norm = sqrt(sum g^2) over every gradient, coef = min(1, max_norm /
    (norm + 1e-6)), g *= coef in place; returns the pre-clip norm (torch's formula, norm type 2)."""
    norm = math.sqrt(sum(float((g.double() * g.double()).sum()) for g in grads))
    coef = min(1.0, max_norm / (norm + 1e-6)) if not math.isnan(norm) else math.nan
    for g in grads:
        g.mul_(coef)
    return norm


@pytest.mark.parametrize("cls", ["fused", "dp"])
def test_constructors_accept_none_numbers_and_inf(cls):
    from rawaudiovae_kelsey_b200.dist import DataParallelTrainStep
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    make = FusedTrainStep if cls == "fused" else DataParallelTrainStep
    assert make(None, None, 0.5).max_grad_norm is None
    assert make(None, None, 0.5, max_grad_norm=1).max_grad_norm == 1.0
    assert make(None, None, 0.5, max_grad_norm=0.25).max_grad_norm == 0.25
    assert make(None, None, 0.5, max_grad_norm=math.inf).max_grad_norm == math.inf
    assert make(None, None, 0.5, max_grad_norm=1.0).grad_norm is None      # no step yet: nothing touched the GPU


@pytest.mark.parametrize("cls", ["fused", "dp"])
@pytest.mark.parametrize("bad", BAD, ids=[repr(b) for b in BAD])
def test_constructors_reject_bad_values_before_gpu_work(cls, bad):
    from rawaudiovae_kelsey_b200.dist import DataParallelTrainStep
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    make = FusedTrainStep if cls == "fused" else DataParallelTrainStep
    with pytest.raises(ValueError, match="max_grad_norm"):
        make(None, None, 0.5, max_grad_norm=bad)


def test_setter_validates():
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    step = FusedTrainStep(None, None, 0.5, max_grad_norm=1.0)
    step.max_grad_norm = 3.0
    assert step.max_grad_norm == 3.0
    step.max_grad_norm = None
    assert step.max_grad_norm is None
    with pytest.raises(ValueError):
        step.max_grad_norm = -2.0
    assert step.max_grad_norm is None


def _cfg(path, **training):
    cfg = configparser.ConfigParser()
    cfg.read(ROOT / path)
    for k, v in training.items():
        cfg["training"][k] = str(v)
    return cfg


@pytest.mark.parametrize("path", ["default.ini", "kelsey_iterable.ini"])
def test_ini_key(path):
    from rawaudiovae_kelsey_b200.trainer import _max_grad_norm
    assert _max_grad_norm(_cfg(path)) is None
    assert _max_grad_norm(_cfg(path, max_grad_norm="")) is None
    assert _max_grad_norm(_cfg(path, max_grad_norm="1.0")) == 1.0
    assert _max_grad_norm(_cfg(path, max_grad_norm="0.5")) == 0.5
    assert _max_grad_norm(_cfg(path, max_grad_norm="inf")) == math.inf
    for bad in ("0", "-1", "nan", "-inf", "one", "1.0.0"):
        with pytest.raises(ValueError, match="max_grad_norm"):
            _max_grad_norm(_cfg(path, max_grad_norm=bad))


@pytest.mark.parametrize("scale", [1e-3, 1.0, 1e3])
@pytest.mark.parametrize("max_norm", [0.5, 1.0, 1e9, math.inf])
def test_reference_agrees_with_torch(scale, max_norm):
    gen = torch.Generator().manual_seed(0)
    shapes = [(64, 32), (32,), (16, 64), (8,), (5, 7)]
    grads = [torch.randn(s, generator=gen, dtype=torch.float64) * scale for s in shapes]
    params = [torch.zeros(s, dtype=torch.float64, requires_grad=True) for s in shapes]
    for p, g in zip(params, grads):
        p.grad = g.clone()
    want = torch.nn.utils.clip_grad_norm_(params, max_norm)
    got = clip_grad_norm(grads, max_norm)
    assert got == pytest.approx(float(want), rel=1e-14)
    for p, g in zip(params, grads):
        assert torch.allclose(p.grad, g, rtol=1e-14, atol=0.0)


def test_reference_propagates_non_finite_norms_like_torch():
    for bad in (math.inf, math.nan):
        g = torch.tensor([1.0, bad], dtype=torch.float64)
        p = torch.zeros(2, dtype=torch.float64, requires_grad=True)
        p.grad = g.clone()
        want = float(torch.nn.utils.clip_grad_norm_([p], 1.0))
        got = clip_grad_norm([g], 1.0)
        assert (math.isnan(got) and math.isnan(want)) or got == want
        assert torch.equal(torch.isnan(g), torch.isnan(p.grad))


def test_entries_are_declared_and_check_arguments_before_the_plan():
    lib = _lib.load()
    assert "rvae_plan_set_grad_clip" in _lib.SIGNATURES and "rvae_plan_grad_norm" in _lib.SIGNATURES
    hdr = (ROOT / "include" / "rvae_b200.h").read_text()
    assert "int rvae_plan_set_grad_clip(rvae_plan* plan, const double* max_norm_dev, float* norm_out, int ring_size);" \
        in hdr
    assert "int rvae_plan_grad_norm(rvae_plan* plan, float* norm_out, void* stream);" in hdr
    # a non-null norm ring of size < 1 is refused before the (bogus) plan pointer is read
    assert lib.rvae_plan_set_grad_clip(8, 8, 8, 0) == 1
    assert b"ring_size" in lib.rvae_last_error()
    assert lib.rvae_plan_set_grad_clip(None, 8, None, 1) == 1
    assert lib.rvae_plan_grad_norm(8, None, None) == 1
    assert b"grad_norm" in lib.rvae_last_error()
    assert lib.rvae_plan_grad_norm(None, 8, None) == 1
    assert lib.rvae_abi_version() == 5
