"""Deterministic training steps without a GPU: the trainers' [training] deterministic and seed keys, the step
constructors' checks, the data-parallel backend refusal, and the C entries with their ctypes signatures."""
import configparser
import ctypes as C
import random

import pytest
import torch

from rawaudiovae_kelsey_b200 import _lib


def _config(**training):
    cfg = configparser.ConfigParser()
    cfg.read_dict({"training": training})
    return cfg


@pytest.mark.parametrize("value, want", [("True", True), ("true", True), ("yes", True), ("1", True),
                                         ("False", False), ("no", False), ("0", False), ("", False)])
def test_ini_deterministic(value, want):
    from rawaudiovae_kelsey_b200.trainer import _deterministic
    assert _deterministic(_config(deterministic=value)) is want
    assert _deterministic(_config()) is False


@pytest.mark.parametrize("value", ["maybe", "2", "on off"])
def test_ini_deterministic_rejects_non_booleans(value):
    from rawaudiovae_kelsey_b200.trainer import _deterministic
    with pytest.raises(ValueError, match="deterministic"):
        _deterministic(_config(deterministic=value))


def test_ini_seed():
    from rawaudiovae_kelsey_b200.trainer import _apply_seed, _seed
    assert _seed(_config()) is None
    assert _seed(_config(seed="")) is None
    assert _seed(_config(seed="0")) == 0
    assert _seed(_config(seed=" 1234 ")) == 1234
    for bad in ("1.5", "zero", "0x10"):
        with pytest.raises(ValueError, match="seed"):
            _seed(_config(seed=bad))
    _apply_seed(7)
    a = (torch.rand(3), random.random())
    _apply_seed(7)
    b = (torch.rand(3), random.random())
    assert torch.equal(a[0], b[0]) and a[1] == b[1]


@pytest.mark.parametrize("path", ["default.ini", "kelsey_iterable.ini"])
def test_ini_files_document_both_keys(path):
    from pathlib import Path
    text = (Path(__file__).resolve().parents[1] / path).read_text()
    assert "# deterministic = True" in text and "# seed = 0" in text
    cfg = configparser.ConfigParser()
    cfg.read_string(text)
    assert "deterministic" not in cfg["training"] and "seed" not in cfg["training"]   # off unless set


@pytest.mark.parametrize("cls", ["fused", "dp"])
def test_constructors(cls):
    from rawaudiovae_kelsey_b200.dist import DataParallelTrainStep
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    make = FusedTrainStep if cls == "fused" else DataParallelTrainStep
    assert make(None, None, 0.5).deterministic is False
    assert make(None, None, 0.5, deterministic=True).deterministic is True
    for bad in (1, 0, "True", None, 1.0, [True]):
        with pytest.raises(ValueError, match="deterministic"):
            make(None, None, 0.5, deterministic=bad)


@pytest.mark.parametrize("backend", ["nvls", "nccl"])
def test_dp_refuses_a_forced_unordered_backend(backend, monkeypatch):
    from rawaudiovae_kelsey_b200.dist import DataParallelTrainStep
    monkeypatch.setenv("RVAE_DP_BACKEND", backend)
    with pytest.raises(ValueError, match=backend):
        DataParallelTrainStep(None, None, 0.5, deterministic=True)
    assert DataParallelTrainStep(None, None, 0.5).deterministic is False   # the default mode is unaffected
    monkeypatch.setenv("RVAE_DP_BACKEND", "p2p")
    assert DataParallelTrainStep(None, None, 0.5, deterministic=True).deterministic is True


def test_abi_symbols_and_signatures():
    lib = _lib.load()
    assert _lib.SIGNATURES["rvae_plan_deterministic_bytes"] == (C.c_size_t, [C.c_void_p])
    assert _lib.SIGNATURES["rvae_plan_set_deterministic"] == (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t])
    assert lib.rvae_plan_deterministic_bytes.restype is C.c_size_t
    assert lib.rvae_abi_version() == 5
    # null plans: 0 bytes, and RVAE_ERR_INVALID before anything touches a device
    assert lib.rvae_plan_deterministic_bytes(None) == 0
    assert lib.rvae_plan_set_deterministic(None, None, 0) == 1
    assert b"null" in lib.rvae_last_error()


# ------------------------------------------------------------------------------------------------ world-2 gloo
def _free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


CASES = [("p2p", "p2p"), ("p2p", "nccl"), ("nvls", "nvls"), ("nccl", "nvls")]


def _gloo_worker(rank, world, port, ret):
    import os
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from rawaudiovae_kelsey_b200 import dist as rdist
    rdist.init_from_env("gloo")
    out = []
    for case in CASES:
        try:
            rdist.agree_peer_loads(case[rank])
            out.append(None)
        except ValueError as e:
            out.append(str(e))
    # a forced unordered backend on a real group: every rank refuses at construction
    forced = []
    for backend in ("nvls", "nccl"):
        os.environ["RVAE_DP_BACKEND"] = backend
        try:
            rdist.DataParallelTrainStep(None, None, 0.5, deterministic=True)
            forced.append(None)
        except ValueError as e:
            forced.append(str(e))
    os.environ["RVAE_DP_BACKEND"] = "auto"
    step = rdist.DataParallelTrainStep(None, None, 0.5, deterministic=True)
    ret.put((rank, out, forced, step.world, step.deterministic))
    dist.barrier()
    dist.destroy_process_group()


def test_dp_backend_refusal_on_a_world_2_gloo_group():
    """Every rank refuses deterministic training unless every rank's gradients go through peer loads, and names the
    other backends; a forced NVLS / NCCL backend refuses at construction on every rank."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(ret.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(60)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    for rank, out, forced, world, det in res:
        assert world == 2 and det is True
        assert out[0] is None, (rank, out[0])
        assert "nccl" in out[1] and "nvls" in out[2] and "nccl" in out[3] and "nvls" in out[3], (rank, out)
        assert "RVAE_DP_BACKEND=nvls" in forced[0] and "RVAE_DP_BACKEND=nccl" in forced[1], (rank, forced)
