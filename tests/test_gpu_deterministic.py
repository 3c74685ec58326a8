"""Deterministic training steps on the GPU (FusedTrainStep(deterministic=True)): two runs give the same bits, whatever
the SM budget, the stage-1 weight-gradient grid, fused or separate launches, graph replay or eager steps; a
deterministic step passes the per-element fp64 check of every launch and issues exactly the default step's launches
plus one gradient-sum launch per bucket."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
DEFAULT = (1024, 2048, 256)
PADDED = (1000, 300, 16)
HOP = 128
CLIP = dict(clip=1e-4, schedule=dict(lr_schedule="cosine", warmup_steps=2, total_steps=20, lr_min=1e-5,
                                     kl_anneal="cyclical", kl_beta_start=0.0, kl_cycles=2, kl_cycle_ratio=0.9))
# name -> (dims, precision, batch sizes in call order, frames read in place, extra step arguments)
RUNS = {
    "default_bf16_8192": (DEFAULT, "bf16", [8192] * 6, False, {}),
    "default_fp32_8192": (DEFAULT, "fp32", [8192] * 6, False, {}),
    "in_place_4096": (DEFAULT, "bf16", [4096] * 6, True, {}),
    "ragged_8155_after_8192": (DEFAULT, "bf16", [8192] * 3 + [8155] * 7, False, {}),
    "padded": (PADDED, "bf16", [200] * 6, False, {}),
    "clip_cosine_cyclical": (DEFAULT, "bf16", [8192] * 6, False, CLIP),
}
STATE = ("params", "exp_avg", "exp_avg_sq", "shadow_hi", "shadow_lo", "step")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def run(name, dev, graph=True, deterministic=True):
    """A fresh seeded model trained on the run's batches with graph replay and next-batch prefetch, as the trainers
    and bench.py do. Returns every output a step covers, on the CPU."""
    from oracle.rawvae_oracle import synth_wav
    from rawaudiovae_kelsey_b200.model import VAE, FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from rawaudiovae_kelsey_b200.schedule import Schedule
    dims, precision, sizes, in_place, extra = RUNS[name]
    S = dims[0]
    torch.manual_seed(0)
    model = VAE(*dims, precision=precision).to(dev)
    model.eps_seed = 5
    opt = Adam(model.parameters(), lr=1e-4)
    step = FusedTrainStep(model, opt, 1e-4, graph=graph, schedule=Schedule(**extra.get("schedule", {})),
                          max_grad_norm=extra.get("clip"), deterministic=deterministic)
    n_frames = 3 * max(sizes) + 64
    audio = torch.from_numpy(synth_wav(np.random.default_rng(3), (n_frames - 1) * HOP + S)).to(dev)
    gen = torch.Generator().manual_seed(21)

    def batch(size, i):
        if in_place:
            return FrameBatch(audio, size, HOP, S, first_frame=(i * 997) % (n_frames - size))
        return FrameBatch(audio, size, HOP, S, frame_idx=torch.randint(0, n_frames, (size,), generator=gen).to(dev))

    batches = [batch(s, i) for i, s in enumerate(sizes)] + [batch(sizes[-1], len(sizes))]
    for i in range(len(sizes)):
        step(batches[i], next_data=batches[i + 1])
    torch.cuda.synchronize()
    flat = model._flat
    out = {k: (getattr(flat, k).cpu() if getattr(flat, k) is not None else None) for k in STATE}
    out["ring"] = step.ring.cpu()
    if step.norm_ring is not None:
        out["norm_ring"] = step.norm_ring.cpu()
    if flat.S != S or flat.H != dims[1] or flat.L != dims[2]:
        out["padding"] = _padding(flat)
    out["stats"] = dict(step.stats)
    return out


def _padding(flat):
    true = torch.zeros(flat.total, dtype=torch.bool, device=flat.params.device)
    for name in flat.geometry:
        flat.view(true, name).fill_(True)
    return {k: int((getattr(flat, k)[~true] != 0).sum()) for k in ("params", "exp_avg", "exp_avg_sq")}


def assert_same_bits(a, b, label):
    for k, v in a.items():
        if k == "stats":
            continue
        if k == "padding":
            assert v == b[k] and not any(v.values()), (label, v, b[k])
            continue
        if v is None:
            assert b[k] is None, (label, k)
            continue
        if k == "ring":   # only the slots of the steps that ran
            v, w = v[:len(RUNS[label][2])], b[k][:len(RUNS[label][2])]
        else:
            w = b[k]
        assert torch.equal(v, w), f"{label}: {k} differs ({int((v != w).sum())} elements)"


@pytest.mark.parametrize("name", list(RUNS))
def test_two_runs_give_the_same_bits(name, dev):
    a, b = run(name, dev), run(name, dev)
    assert a["stats"]["replays"] >= 2, a["stats"]
    assert_same_bits(a, b, name)
    assert bool(torch.isfinite(a["params"]).all())


_CHILD = """
import sys, torch
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
from test_gpu_deterministic import run
out = run({name!r}, torch.device("cuda", 0))
torch.save(out, {path!r})
"""


@pytest.mark.parametrize("env", [{"RVAE_NUM_SMS": "128", "RVAE_S1_WGRAD_CTAS": "64"}, {"RVAE_DUAL_PAIRS": "0"}],
                         ids=["sm_budget", "separate_launches"])
@pytest.mark.parametrize("name", ["default_bf16_8192", "ragged_8155_after_8192"])
def test_bits_do_not_depend_on_scheduling(name, env, dev, tmp_path):
    """The same run in a process with a smaller SM budget and stage-1 grid, or with every fused backward launch split
    into separate GEMMs, gives the bits of the run in this process."""
    path = tmp_path / "out.pt"
    code = _CHILD.format(root=str(ROOT), tests=str(ROOT / "tests"), name=name, path=str(path))
    res = subprocess.run([sys.executable, "-c", code], env={**os.environ, **env}, cwd=str(ROOT),
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    assert_same_bits(run(name, dev), torch.load(path), name)


def test_eager_steps_equal_replayed_steps(dev):
    eager = run("default_bf16_8192", dev, graph=False)
    assert eager["stats"]["replays"] == 0
    assert_same_bits(eager, run("default_bf16_8192", dev), "default_bf16_8192")


def test_deterministic_agrees_with_the_default_step(dev):
    """Same seed and data, deterministic against default: the same update up to the last bits of reordered sums."""
    det, ref = run("default_bf16_8192", dev), run("default_bf16_8192", dev, deterministic=False)
    for k in ("params", "exp_avg", "exp_avg_sq"):
        a, b = det[k].double(), ref[k].double()
        assert float((a - b).norm() / b.norm()) < 1e-2, k
    assert torch.allclose(det["ring"], ref["ring"], rtol=1e-3, atol=0), (det["ring"][:6], ref["ring"][:6])


@pytest.mark.parametrize("name", ["default_gather_bf16", "default_gather_fp32", "default_ragged_8155_after_8192",
                                  "padded_b200", "small_b129", "default_clip_cosine_cyclical"])
def test_deterministic_step_every_launch_elementwise(name, dev, monkeypatch):
    """The per-element fp64 check of every launch of a deterministic step; its eager step launches the default
    step's kernels plus one gradient-sum launch per bucket (4)."""
    import test_gpu_step_elementwise as E
    from rawaudiovae_kelsey_b200 import model as M
    base = M.FusedTrainStep

    class DetStep(base):
        def __init__(self, *a, **k):
            super().__init__(*a, deterministic=True, **k)

    monkeypatch.setattr(M, "FusedTrainStep", DetStep)
    expected = E.expected_launches
    monkeypatch.setattr(E, "expected_launches", lambda case: expected(case) + 4)
    checkers = E.run_case(name, dev)
    E._report(checkers)
    failures = [f for ck in checkers for f in ck.failures]
    assert not failures, "\n".join(failures[:40])


# ------------------------------------------------------------------------------------------------ trainers
TRAINERS = [
    ("epoch", (1024, 256, 64), 128, 512, "epochs = 3\nsave_best_model_after = 1\ncheckpoint_interval = 1"),
    ("stream", (1024, 256, 64), 128, 256, "epochs = 1\ntotal_num_frames = 2560\ncheckpoint_interval = 4\n"
                                           "log_interval = 3"),
]


def _train(tmp, which, dims, hop, batch, extra, rng_seed):
    """One trainer run with [training] deterministic = True and seed = 0. The process RNGs are first set to
    `rng_seed`, so only the seed key can make two runs start alike."""
    import random
    from test_gpu_parity import _trainer_ini
    from test_gpu_param_histograms import _corpus
    from rawaudiovae_kelsey_b200 import trainer
    data = _corpus(tmp)
    ini = tmp / "t.ini"
    _trainer_ini(ini, data, batch=batch, extra_training=extra + "\ndeterministic = True\nseed = 0")
    S, H, L = dims
    text = ini.read_text()
    for a, b in (("hop_length = 128", f"hop_length = {hop}"), ("segment_length = 1024", f"segment_length = {S}"),
                 ("latent_dim = 64", f"latent_dim = {L}"), ("n_units = 256", f"n_units = {H}")):
        text = text.replace(a, b)
    ini.write_text(text)
    torch.manual_seed(rng_seed)
    random.seed(rng_seed)
    fn = trainer.run_epoch_trainer if which == "epoch" else trainer.run_stream_trainer
    assert fn(["--config", str(ini)]) in (0, None)
    return next((data / "unit-test").glob("run-*"))


@pytest.mark.parametrize("cfg", TRAINERS, ids=lambda c: c[0])
def test_trainer_runs_are_bitwise_equal(cfg, dev, tmp_path):
    """Two runs of a trainer with deterministic = True and seed = 0: bitwise equal checkpoints, test_reconst_*.wav
    files and Loss/Batch scalars."""
    from test_gpu_eval import _same_run, _scalars
    which, dims, hop, batch, extra = cfg
    a = _train(tmp_path / "a", which, dims, hop, batch, extra, rng_seed=11)
    b = _train(tmp_path / "b", which, dims, hop, batch, extra, rng_seed=12)
    assert len(list((a / "model" / "checkpoints").glob("ckpt_*"))) >= 2
    assert list((a / "audio_logs").glob("test_reconst_*.wav"))
    assert _same_run(a, b) and _same_run(b, a)
    la, lb = _scalars(a)["Loss/Batch"], _scalars(b)["Loss/Batch"]
    assert la and la == lb, (la, lb)


# ------------------------------------------------------------------------------------------------ data parallel
def _free_port():
    import socket
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    port = sk.getsockname()[1]
    sk.close()
    return port


def _dp_worker(rank, world, port, ret):
    """One rank: two deterministic DataParallelTrainStep runs from the same weights on the same shards (graph=True,
    Philox noise); the run's parameters, moments, step counter and loss ring, and the replica on rank 0."""
    sys.path.insert(0, str(ROOT))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from rawaudiovae_kelsey_b200 import dist as rdist
    from rawaudiovae_kelsey_b200.dataset import shard_bounds
    from rawaudiovae_kelsey_b200.model import VAE
    from rawaudiovae_kelsey_b200.optim import Adam
    _, _, local = rdist.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    S, H, L, B, n = 1024, 2048, 256, 8192, 6
    gen = torch.Generator().manual_seed(1)
    xs = [(torch.rand(B, S, generator=gen) * 2 - 1).to(dev) for _ in range(2)]
    lo, hi = shard_bounds(B, rank, world)

    def one_run():
        torch.manual_seed(0)
        m = VAE(S, H, L).to(dev)
        m.eps_seed = 123
        step = rdist.DataParallelTrainStep(m, Adam(m.parameters(), lr=1e-4), 1e-4, global_batch=B, graph=True,
                                           deterministic=True)
        for i in range(n):
            step(xs[i % 2][lo:hi].contiguous())
        torch.cuda.synchronize()
        f = m._flat
        return {"params": f.params.clone(), "exp_avg": f.exp_avg.clone(), "exp_avg_sq": f.exp_avg_sq.clone(),
                "step": f.step.clone(), "ring": step.ring[:n].clone(), "replays": step.stats["replays"]}

    a, b = one_run(), one_run()
    runs_equal = all(torch.equal(a[k], b[k]) for k in ("params", "exp_avg", "exp_avg_sq", "step", "ring"))
    ref = a["params"].clone()
    dist.broadcast(ref, src=0)
    replicas_equal = bool(torch.equal(ref, a["params"]))
    os.environ["RVAE_DP_BACKEND"] = "nccl"
    try:
        rdist.DataParallelTrainStep(None, None, 1e-4, deterministic=True)
        refused = False
    except ValueError:
        refused = True
    ret.put((rank, runs_equal, replicas_equal, refused, a["replays"]))
    dist.barrier()
    dist.destroy_process_group()


def test_data_parallel_runs_and_replicas_are_bitwise_equal(dev):
    """2 ranks, deterministic: two runs give the same bits, the replicas are bitwise equal, and a forced NCCL exchange
    is refused at construction."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs: the data-parallel step runs one rank per GPU")
    import queue
    import time
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    out, deadline = [], time.monotonic() + 600
    while len(out) < 2:
        try:
            out.append(ret.get(timeout=5))
        except queue.Empty:
            if any(p.exitcode not in (None, 0) for p in procs) or time.monotonic() > deadline:
                for p in procs:
                    p.kill()
                raise AssertionError(f"a rank failed: exit codes {[p.exitcode for p in procs]}")
    for p in procs:
        p.join(120)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    for rank, runs_equal, replicas_equal, refused, replays in sorted(out):
        assert replays > 0 and runs_equal and replicas_equal and refused, (rank, runs_equal, replicas_equal, refused)
