"""Learning-rate and KL-weight schedules without a GPU: the host mirror at known steps, validation, the rvae_hparams
record against the header and rvae_hparams_check, and the trainers' ini keys."""
import configparser
import ctypes as C
import math
import re
from pathlib import Path

import pytest

from rawaudiovae_kelsey_b200 import _lib
from rawaudiovae_kelsey_b200.schedule import Schedule, _cos_pi_unit

ROOT = Path(__file__).resolve().parents[1]
LR = 1e-3


def test_cos_polynomial_is_cos():
    for i in range(101):
        u = i / 100
        assert abs(_cos_pi_unit(u) - math.cos(math.pi * u)) < 4e-16
    assert _cos_pi_unit(0.0) == 1.0 and _cos_pi_unit(1.0) == -1.0 and abs(_cos_pi_unit(0.5)) < 1e-16


def test_constant_schedule_is_the_peak_value_at_every_step():
    s = Schedule()
    for k in (0, 1, 10, 10 ** 6):
        assert s.lr_at(k, LR) == LR
        assert s.beta_at(k, 1e-4) == 1e-4


def test_warmup():
    s = Schedule(warmup_steps=4)
    assert [s.lr_at(k, LR) for k in range(6)] == [LR * 1 / 4, LR * 2 / 4, LR * 3 / 4, LR, LR, LR]


@pytest.mark.parametrize("kind", ["linear", "cosine"])
def test_decay_at_boundaries(kind):
    W, T, lo = 10, 110, 1e-5
    s = Schedule(lr_schedule=kind, warmup_steps=W, total_steps=T, lr_min=lo)
    assert s.lr_at(0, LR) == LR / W
    assert s.lr_at(W - 1, LR) == LR * W / W
    assert s.lr_at(W, LR) == pytest.approx(LR, rel=1e-15)
    assert s.lr_at(T, LR) == pytest.approx(lo, rel=1e-12)
    assert s.lr_at(T + 10 ** 4, LR) == s.lr_at(T, LR)          # steps past T hold the final value
    assert lo < s.lr_at(T - 1, LR) < s.lr_at(W + 1, LR) < LR
    mid = s.lr_at(W + (T - W) // 2, LR)                          # u = 0.5
    assert mid == pytest.approx(lo + (LR - lo) * 0.5, rel=1e-15)
    if kind == "cosine":
        u = 0.25
        assert s.lr_at(W + 25, LR) == pytest.approx(lo + (LR - lo) * 0.5 * (1 + math.cos(math.pi * u)), rel=1e-15)


def test_linear_kl_annealing():
    s = Schedule(kl_anneal="linear", kl_beta_start=0.0, kl_anneal_steps=100)
    assert s.beta_at(0, 1.0) == 0.0
    assert s.beta_at(50, 1.0) == 0.5
    assert s.beta_at(100, 1.0) == 1.0 and s.beta_at(10 ** 5, 1.0) == 1.0


def test_cyclical_kl_annealing_cycle_boundaries():
    # T = 100, M = 3 -> C = 34; ramp over the first half of each cycle
    s = Schedule(kl_anneal="cyclical", total_steps=100, kl_cycles=3, kl_cycle_ratio=0.5, kl_beta_start=0.1)
    assert s.beta_at(0, 1.0) == 0.1
    assert s.beta_at(17, 1.0) == 1.0 and s.beta_at(33, 1.0) == 1.0
    assert s.beta_at(34, 1.0) == 0.1 and s.beta_at(68, 1.0) == 0.1
    assert s.beta_at(34 + 8, 1.0) == pytest.approx(0.1 + 0.9 * (8 / 34 / 0.5), rel=1e-15)


@pytest.mark.parametrize("kw, words", [
    (dict(lr_schedule="step"), "lr_schedule"), (dict(kl_anneal="sigmoid"), "kl_anneal"),
    (dict(warmup_steps=-1), "warmup_steps"), (dict(lr_schedule="cosine", total_steps=0), "total_steps"),
    (dict(lr_schedule="linear"), "total_steps"), (dict(kl_anneal="cyclical", total_steps=0), "total_steps"),
    (dict(kl_anneal="linear", kl_anneal_steps=0), "kl_anneal_steps"),
    (dict(kl_anneal="cyclical", total_steps=10, kl_cycles=0), "kl_cycles"),
    (dict(kl_cycle_ratio=0.0), "kl_cycle_ratio"), (dict(kl_cycle_ratio=1.5), "kl_cycle_ratio"),
    (dict(lr_min=float("nan")), "lr_min"), (dict(kl_beta_start=float("inf")), "kl_beta_start"),
    (dict(warmup_steps=2.5), "warmup_steps"),
])
def test_validation_errors(kw, words):
    with pytest.raises(ValueError, match=words):
        Schedule(**kw)


def test_record_rejects_non_finite_peak_values():
    with pytest.raises(ValueError, match="lr"):
        Schedule().record(float("inf"), (0.9, 0.999), 1e-8, 0.0, 1e-4)
    with pytest.raises(ValueError, match="kl_beta"):
        Schedule().record(1e-4, (0.9, 0.999), 1e-8, 0.0, float("nan"))


def test_record_layout_matches_the_header():
    hdr = (ROOT / "include" / "rvae_b200.h").read_text()
    body = re.search(r"typedef struct rvae_hparams \{(.*?)\} rvae_hparams;\s*/\* (\d+) bytes", hdr, re.S)
    assert body is not None
    fields = re.findall(r"^\s*(double|int64_t|int32_t) (\w+);\s*/\*\s*(\d+)", body.group(1), re.M)
    assert [(n, int(o)) for _, n, o in fields] == [(n, getattr(_lib.Hparams, n).offset) for n, _ in
                                                   _lib.Hparams._fields_]
    sizes = {"double": 8, "int64_t": 8, "int32_t": 4}
    assert [sizes[t] for t, _, _ in fields] == [getattr(_lib.Hparams, n).size for n, _ in _lib.Hparams._fields_]
    assert C.sizeof(_lib.Hparams) == int(body.group(2)) == 112


def _raw(**over):
    base = dict(lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, kl_beta=1e-4, lr_min=0.0,
                kl_beta_start=0.0, kl_cycle_ratio=0.5, total_steps=0, warmup_steps=0, kl_anneal_steps=1, kl_cycles=1,
                lr_schedule=0, kl_anneal=0)
    base.update(over)
    return _lib.Hparams(**base)


KINDS_LR = {"constant": 0, "linear": 1, "cosine": 2}
KINDS_KL = {"constant": 0, "linear": 1, "cyclical": 2}
CASES = [
    dict(), dict(lr_schedule="cosine", total_steps=10, warmup_steps=3), dict(lr_schedule="linear", total_steps=1),
    dict(lr_schedule="cosine", total_steps=0), dict(lr_schedule="linear", total_steps=-5), dict(warmup_steps=-1),
    dict(kl_anneal="linear", kl_anneal_steps=0), dict(kl_anneal="linear", kl_anneal_steps=5),
    dict(kl_anneal="cyclical", total_steps=10, kl_cycles=0), dict(kl_anneal="cyclical", total_steps=0),
    dict(kl_anneal="cyclical", total_steps=10, kl_cycles=4, kl_cycle_ratio=1.0),
    dict(kl_cycle_ratio=0.0), dict(kl_cycle_ratio=-0.5), dict(kl_cycle_ratio=1.0000001), dict(lr_min=float("inf")),
    dict(kl_beta_start=float("nan")), dict(kl_anneal_steps=0), dict(kl_cycles=-3), dict(total_steps=-1),
]


@pytest.mark.parametrize("case", CASES, ids=[str(c) for c in CASES])
def test_check_agrees_with_schedule_validation(case):
    lib = _lib.load()
    try:
        Schedule(**case)
        ok = True
    except ValueError:
        ok = False
    raw = dict(case)
    raw["lr_schedule"] = KINDS_LR[raw.get("lr_schedule", "constant")]
    raw["kl_anneal"] = KINDS_KL[raw.get("kl_anneal", "constant")]
    assert (lib.rvae_hparams_check(C.byref(_raw(**raw))) == 0) == ok, lib.rvae_last_error()


@pytest.mark.parametrize("over", [dict(lr_schedule=3), dict(lr_schedule=-1), dict(kl_anneal=3),
                                  dict(lr=float("nan")), dict(beta2=float("inf")), dict(eps=float("nan")),
                                  dict(weight_decay=float("-inf")), dict(kl_beta=float("nan"))])
def test_check_refuses_what_schedule_cannot_express(over):
    assert _lib.load().rvae_hparams_check(C.byref(_raw(**over))) == 1


def test_device_entries_reject_bad_arguments_before_the_context():
    lib = _lib.load()
    assert lib.rvae_hparams_eval(None, None, 8, 1, 8, 8, None) == 1
    assert lib.rvae_hparams_eval(None, 8, 8, 0, 8, 8, None) == 1
    assert b"hparams_eval" in lib.rvae_last_error()
    assert lib.rvae_plan_train_step_hp(None, None, 1, None, 1, None) == 1
    assert lib.rvae_plan_train_step_hp(None, 8, 1, None, 0, None) == 1
    assert b"train_step_hp" in lib.rvae_last_error()
    assert lib.rvae_abi_version() == 5


def _cfg(path, **keys):
    cfg = configparser.ConfigParser()
    cfg.read(ROOT / path)
    for k, v in keys.items():
        sec, name = k.split("__")
        cfg[sec][name] = str(v)
    return cfg


@pytest.mark.parametrize("path", ["default.ini", "kelsey_iterable.ini"])
def test_default_keys_give_the_constant_schedule(path):
    from rawaudiovae_kelsey_b200.trainer import _schedule
    s = _schedule(_cfg(path), 1000)
    assert s.lr_schedule == "constant" and s.kl_anneal == "constant" and s.warmup_steps == 0
    assert s.lr_at(0, 1e-4) == 1e-4 and s.lr_at(999, 1e-4) == 1e-4 and s.beta_at(5, 1e-4) == 1e-4


def test_ini_keys_are_parsed():
    from rawaudiovae_kelsey_b200.trainer import _schedule
    s = _schedule(_cfg("kelsey_iterable.ini", training__lr_schedule="cosine", training__lr_warmup_steps=50,
                       training__lr_min=1e-6, VAE__kl_anneal="cyclical", VAE__kl_beta_start=0.0, VAE__kl_cycles=4,
                       VAE__kl_cycle_ratio=0.25), 37674)
    assert s == Schedule("cosine", 50, 37674, 1e-6, "cyclical", 0.0, 37674, 4, 0.25)
    with pytest.raises(ValueError, match="lr_schedule"):
        _schedule(_cfg("default.ini", training__lr_schedule="exp"), 10)
    with pytest.raises(ValueError):
        _schedule(_cfg("default.ini", training__lr_warmup_steps="many"), 10)


def test_total_steps_of_both_trainers():
    from rawaudiovae_kelsey_b200.trainer import _epoch_trainer_steps, _stream_trainer_steps
    # default.ini: 500 epochs of batch 131072
    cfg = _cfg("default.ini")
    assert _epoch_trainer_steps(cfg, 1_000_000) == 500 * 8
    assert _epoch_trainer_steps(cfg, 131072 * 3) == 500 * 3
    assert _epoch_trainer_steps(cfg, 131072 * 3 + 1) == 500 * 4
    assert _epoch_trainer_steps(cfg, 131072 * 3 + 1, world=2) == 500 * 3   # a 1-frame last batch is skipped on 2 ranks
    assert _epoch_trainer_steps(cfg, 131072 * 3 + 2, world=2) == 500 * 4
    assert _epoch_trainer_steps(_cfg("default.ini", training__epochs=2, training__batch_size=100), 1001) == 22
    # kelsey_iterable.ini: total_num_frames / batch_size, truncated
    assert _stream_trainer_steps(_cfg("kelsey_iterable.ini")) == 154314100 // 4096 == 37674
    assert _stream_trainer_steps(_cfg("kelsey_iterable.ini", training__total_num_frames=1000,
                                      training__batch_size=300)) == 3
