"""Scheduled learning rate and KL weight on the GPU: the device function against the host mirror, Adam at lr(k),
CUDA-graph replays that follow the schedule (against the fp64 oracle) and host-side changes, resume, the 2-rank
data-parallel step and the trainers."""
import os
import random
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import rawvae_oracle as O

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
TOL = {"bf16": 2e-2, "fp32": 1e-4}    # the repository's tolerances against the fp64 oracle


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def make(dims, precision, dev, seed=0):
    from rawaudiovae_kelsey_b200.model import VAE
    p64 = {k: v.double() for k, v in O.init_params(*dims, seed=seed).items()}
    torch.manual_seed(seed)
    m = VAE(*dims, precision=precision)
    m.load_state_dict({k: v.float() for k, v in p64.items()})
    return m.to(dev)


def _upload(rec, dev):
    return torch.frombuffer(bytearray(bytes(rec)), dtype=torch.uint8).to(dev)


SCHEDULES = [
    dict(),
    dict(warmup_steps=7),
    dict(lr_schedule="linear", warmup_steps=10, total_steps=110, lr_min=1e-6),
    dict(lr_schedule="cosine", warmup_steps=10, total_steps=110, lr_min=1e-6),
    dict(lr_schedule="cosine", total_steps=1000, lr_min=0.0),
    dict(kl_anneal="linear", kl_beta_start=1e-6, kl_anneal_steps=37),
    dict(kl_anneal="cyclical", total_steps=110, kl_cycles=3, kl_cycle_ratio=0.4, kl_beta_start=0.0),
]


@pytest.mark.parametrize("kw", SCHEDULES, ids=[str(k) for k in SCHEDULES])
def test_device_equals_host(kw, dev):
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.schedule import Schedule
    s = Schedule(**kw)
    T, W = max(s.total_steps, 1), s.warmup_steps
    ks = sorted({0, 1, max(W - 1, 0), W, W + 1, (T + W) // 2, T - 1, T, T + 1, T + 10 ** 4, 33, 34, 36, 37, 38, 73,
                 2 ** 23, 2 ** 24})
    rec = _upload(s.record(3e-4, (0.9, 0.999), 1e-8, 0.0, 2e-3), dev)
    lr, beta = ops.hparams_eval(rec, torch.tensor(ks, dtype=torch.int64, device=dev))
    want_lr = np.array([s.lr_at(k, 3e-4) for k in ks])
    want_beta = np.array([s.beta_at(k, 2e-3) for k in ks], dtype=np.float32)
    # bitwise, cosine included: the cosine is a fixed polynomial on both sides
    assert np.array_equal(lr.cpu().numpy(), want_lr), (lr.cpu().numpy() - want_lr)
    assert np.array_equal(beta.cpu().numpy(), want_beta)


def _warmup_run(dev, graph, steps=6):
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.schedule import Schedule
    from rawaudiovae_kelsey_b200.optim import Adam
    model = make((1024, 256, 64), "fp32", dev)
    model.eps_seed = 5
    opt = Adam(model.parameters(), lr=1e-3)
    sched = Schedule(warmup_steps=4)
    step = FusedTrainStep(model, opt, kl_beta=0.5, keep_grads=True, graph=graph, schedule=sched)
    x = torch.from_numpy(O.synth_wav(np.random.default_rng(1), 1024 * 256).astype(np.float32)).to(dev)
    x = x.reshape(256, 1024)
    return model, opt, sched, step, x


def test_adam_applies_the_scheduled_lr(dev):
    model, opt, sched, step, x = _warmup_run(dev, graph=False)   # lr(k) = 1/4, 2/4, 3/4, 1, 1, 1 x 1e-3
    flat = model._flat
    for k in range(6):
        p0 = flat.params.clone()
        m0, v0 = flat.exp_avg.clone(), flat.exp_avg_sq.clone()
        step(x)
        torch.cuda.synchronize()
        g = flat.grads.double()

        def host(lr_k):
            t = k + 1
            m = m0.double() + (1 - 0.9) * (g - m0.double())
            v = 0.999 * v0.double() + (1 - 0.999) * g * g
            return p0.double() - lr_k / (1 - 0.9 ** t) * m / (v.sqrt() / (1 - 0.999 ** t) ** 0.5 + 1e-8)
        p1 = flat.params.double()
        scale = float((p1 - p0.double()).abs().max())
        # the kernel rounds the new parameter to fp32: half an ulp of it on top of 1e-6 of the update
        ulp = (torch.nextafter(flat.params.abs(), torch.tensor(float("inf"), device=dev)) - flat.params.abs()).double()
        err = (p1 - host(sched.lr_at(k, 1e-3))).abs()
        assert bool((err <= 1e-6 * scale + 0.5 * ulp).all()), (k, float(err.max()), scale)
        for kk in (k - 1, k + 1):
            if 0 <= kk and sched.lr_at(kk, 1e-3) != sched.lr_at(k, 1e-3):
                other = float((p1 - host(sched.lr_at(kk, 1e-3))).abs().max())
                assert other > 0.1 * scale, (k, kk, other, scale)


@pytest.mark.parametrize("dims, hop, precision", [((1024, 256, 64), 256, "bf16"), ((1024, 256, 64), 256, "fp32"),
                                                  ((1000, 300, 16), 200, "bf16"), ((1000, 300, 16), 200, "fp32")])
def test_graph_replays_follow_the_schedule(dims, hop, precision, dev):
    """Graph + prefetch under a cosine / linear-annealing schedule against the fp64 oracle's train_step driven with
    lr(k), beta(k) and the same Philox noise - parameters after the first three (warm-up) steps and losses of the
    first eight at the repository's few-step tolerances, losses of all 40 steps at its loss-curve tolerance (1 %;
    Adam turns rounding differences of near-zero gradients into whole learning-rate steps, so longer runs part
    ways) - and against eager steps through rvae_plan_train_step, the scalar entry point, with lr and kl_beta set by
    the host before every step."""
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from rawaudiovae_kelsey_b200.schedule import Schedule
    S, L = dims[0], dims[2]
    B, n = 256, 40
    sched = Schedule("cosine", 5, n, 1e-5, "linear", 0.0, 20)
    wav = O.synth_wav(np.random.default_rng(3), hop * (n * B + 20) + S).astype(np.float32)
    audio = torch.from_numpy(wav).to(dev)
    batches = [FrameBatch(audio, B, hop, S, first_frame=i * B) for i in range(n)]

    class ScalarStep(FusedTrainStep):     # the parent's path: every hyper-parameter passed by value
        def _enqueue(self, plan):
            g = self.optimizer.param_groups[0]
            plan.train_step(self.kl_beta, g["lr"], *g["betas"], g["eps"], 0.0, loss_out=self.ring,
                            ring_size=self.ring_size, zero_grads=True)

    def run(scheduled):
        model = make(dims, precision, dev)
        model.eps_seed = 11
        opt = Adam(model.parameters(), lr=1e-3)
        step = (FusedTrainStep(model, opt, kl_beta=0.5, graph=True, schedule=sched) if scheduled
                else ScalarStep(model, opt, kl_beta=0.5))
        losses, early = [], None
        for i, b in enumerate(batches):
            if not scheduled:
                opt.param_groups[0]["lr"] = sched.lr_at(i, 1e-3)
                step.kl_beta = sched.beta_at(i, 0.5)
            nxt = batches[i + 1] if scheduled and i + 1 < n else None
            losses.append(step(b, next_data=nxt).clone())
            if i == 2:
                early = {k: v.detach().clone() for k, v in model.state_dict().items()}
        torch.cuda.synchronize()
        if scheduled:
            assert step.stats["replays"] >= n - 6   # eager and capture calls of both input-set parities
        return torch.stack(losses), model._flat.params.clone(), early

    g_loss, g_par, g_early = run(True)
    # the oracle: step k sees frames k*B.. and the Philox draw at offset k (the device step counter)
    p64 = {k: v.double() for k, v in O.init_params(*dims, seed=0).items()}
    state = O.adam_init(p64)
    frames = torch.from_numpy(O.audio_dataset_frames(wav, S, hop)).double()
    ref, par_err = [], None
    for k in range(n):
        eps = ops.randn((B, L), 11, k, device=dev).double().cpu()
        ref.append(O.train_step(p64, state, frames[k * B:(k + 1) * B], eps, sched.beta_at(k, 0.5),
                                sched.lr_at(k, 1e-3)))
        if k == 2:
            par_err = max(rel(v, p64[name]) for name, v in g_early.items())
    ref = torch.tensor(ref, dtype=torch.float64)
    loss_err = ((g_loss.double().cpu() - ref).abs() / ref.abs())
    # few-step tolerances: losses TOL; parameters after Adam steps 1e-3 in fp32 (test_gpu_padded_dims), TOL in bf16
    assert float(loss_err[:8].max()) <= TOL[precision], loss_err[:8]
    assert par_err <= {"fp32": 1e-3, "bf16": TOL["bf16"]}[precision], par_err
    assert float(loss_err.max()) <= 1e-2, loss_err
    e1_loss, e1_par, _ = run(False)
    e2_loss, e2_par, _ = run(False)
    spread_l, spread_p = rel(e1_loss, e2_loss), rel(e1_par, e2_par)
    # graph + prefetch frames and reduces differently from an eager step (in-place framing, split-K order): the
    # tolerances of test_gpu_padded_dims' graph / prefetch test, or the spread of two eager runs if that is larger
    assert rel(g_loss, e1_loss) <= max(3 * spread_l, 1e-4), (rel(g_loss, e1_loss), spread_l)
    assert rel(g_par, e1_par) <= max(3 * spread_p, 1e-3), (rel(g_par, e1_par), spread_p)
    # the loss ring holds the objective at beta(k): the first steps (beta ~ 0) are mostly reconstruction
    assert torch.isfinite(g_loss).all()


def test_host_changes_reach_replays(dev):
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    model = make((1024, 256, 64), "bf16", dev)
    model.eps_seed = 2
    opt = Adam(model.parameters(), lr=1e-3)
    step = FusedTrainStep(model, opt, kl_beta=0.5, graph=True)
    x = torch.from_numpy(O.synth_wav(np.random.default_rng(2), 1024 * 256).astype(np.float32)).to(dev)
    x = x.reshape(256, 1024)
    for _ in range(3):
        step(x)
    assert step.stats["captures"] == 1
    opt.param_groups[0]["lr"] = 0.0
    flat = model._flat
    torch.cuda.synchronize()
    p0, m0 = flat.params.clone(), flat.exp_avg.clone()
    for _ in range(2):
        step(x)
    torch.cuda.synchronize()
    assert step.stats["replays"] >= 2
    assert torch.equal(flat.params, p0)
    assert not torch.equal(flat.exp_avg, m0)
    # a new kl_beta: the ring's loss of the replay equals the loss of an eager step at that beta
    step.kl_beta = 2.0
    snap = {k: getattr(flat, k).clone() for k in ("params", "exp_avg", "exp_avg_sq", "step")}
    replays = step.stats["replays"]
    got = step(x).clone()
    torch.cuda.synchronize()
    assert step.stats["replays"] == replays + 1     # the new beta reached a replay, not a new capture
    for k, v in snap.items():
        getattr(flat, k).copy_(v)
    flat.sync_shadow()
    eager = FusedTrainStep(model, opt, kl_beta=2.0, graph=False)
    want = eager(x).clone()
    torch.cuda.synchronize()
    assert abs(float(got) - float(want)) <= 1e-5 * abs(float(want)), (float(got), float(want))


def test_resume_continues_the_schedule(dev):
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from rawaudiovae_kelsey_b200.schedule import Schedule
    k0 = 9
    model = make((1024, 256, 64), "bf16", dev)
    model.eps_seed = 4
    opt = Adam(model.parameters(), lr=1e-3)
    x = torch.from_numpy(O.synth_wav(np.random.default_rng(4), 1024 * 256).astype(np.float32)).to(dev)
    x = x.reshape(256, 1024)
    first = FusedTrainStep(model, opt, kl_beta=0.5)
    for _ in range(k0):
        first(x)
    state = opt.state_dict()
    model2 = make((1024, 256, 64), "bf16", dev)
    model2.load_state_dict(model.state_dict())
    model2.eps_seed = 4
    opt2 = Adam(model2.parameters(), lr=1e-3)
    opt2.load_state_dict(state)
    step = FusedTrainStep(model2, opt2, kl_beta=0.5, graph=True,
                          schedule=Schedule("linear", 0, k0, 0.0))
    step(x)      # the first step of the restored run is step k0: lr(k0) = lr_min = 0
    torch.cuda.synchronize()
    assert int(model2._flat.step.item()) == k0 + 1
    for name, p in model2.state_dict().items():
        assert torch.equal(p, model.state_dict()[name]), name


def _free_port():
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    port = sk.getsockname()[1]
    sk.close()
    return port


def _dp_worker(rank, world, port, ret):
    """One rank: the DataParallelTrainStep on its shard and the single-process FusedTrainStep on the whole batch, both
    graph=True with Philox noise under a cosine + cyclical schedule, from identical weights."""
    sys.path.insert(0, str(ROOT))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from rawaudiovae_kelsey_b200 import dist as rdist
    from rawaudiovae_kelsey_b200.dataset import shard_bounds
    from rawaudiovae_kelsey_b200.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from rawaudiovae_kelsey_b200.schedule import Schedule
    _, _, local = rdist.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    S, H, L, B, n = 1024, 256, 64, 1000, 6
    sched = Schedule("cosine", 2, n, 1e-5, "cyclical", 0.0, 1, 2, 0.5)
    gen = torch.Generator().manual_seed(1)
    x = (torch.rand(B, S, generator=gen) * 2 - 1).to(dev)

    def build():
        torch.manual_seed(0)
        m = VAE(S, H, L).to(dev)
        m.eps_seed = 123
        return m, Adam(m.parameters(), lr=1e-3)

    m_dp, o_dp = build()
    m_1, o_1 = build()
    step_dp = rdist.DataParallelTrainStep(m_dp, o_dp, 0.5, global_batch=B, reduce_loss=True, graph=True,
                                          schedule=sched)
    step_1 = FusedTrainStep(m_1, o_1, 0.5, graph=True, schedule=sched)
    lo, hi = shard_bounds(B, rank, world)
    dl = 0.0
    for _ in range(n):
        l_dp = step_dp(x[lo:hi].contiguous())
        l_1 = step_1(x)
        torch.cuda.synchronize()
        dl = max(dl, abs(float(l_dp) - float(l_1)) / float(l_1))
    dw = float((m_dp._flat.params.double() - m_1._flat.params.double()).norm() / m_1._flat.params.double().norm())
    ref = m_dp._flat.params.clone()
    if dist.is_initialized():
        dist.broadcast(ref, src=0)
    same = bool(torch.equal(ref, m_dp._flat.params))
    ret.put((rank, same, dl, dw, step_dp.stats["replays"], step_1.stats["replays"]))
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()


def _run_dp(world):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    import queue
    import time
    out, deadline = [], time.monotonic() + 600
    while len(out) < world:
        try:
            out.append(ret.get(timeout=5))
        except queue.Empty:
            # a rank that died cannot report: stop waiting for it (and stop its peers)
            if any(p.exitcode not in (None, 0) for p in procs) or time.monotonic() > deadline:
                for p in procs:
                    p.kill()
                raise AssertionError(f"a rank failed: exit codes {[p.exitcode for p in procs]}")
    for p in procs:
        p.join(120)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    return sorted(out)


def test_data_parallel_replicas_follow_the_schedule(dev):
    """2 ranks, graph=True, cosine learning rate + cyclical KL weight: the replicas stay bitwise equal, and match the
    single process on the whole batch within tools/dp_check.py's tolerances for Philox steps (loss 1e-4, weights
    4e-3 relative)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs: the data-parallel step runs one rank per GPU")
    for rank, same, dl, dw, rep_dp, rep_1 in _run_dp(2):
        assert rep_dp > 0 and rep_1 > 0, rank
        assert same, rank
        assert dl < 1e-4 and dw < 4e-3, (rank, dl, dw)


def _scalars(run):
    from tensorboard.backend.event_processing.event_file_loader import LegacyEventFileLoader
    out = {}
    for f in sorted((run / "logs").glob("events.out.tfevents.*")):
        for ev in LegacyEventFileLoader(str(f)).Load():
            for v in ev.summary.value:
                out.setdefault(v.tag, {})[ev.step] = v.simple_value if v.HasField("simple_value") else None
    return out


def _write_wavs(root, n_files, seconds, seed):
    from scipy.io import wavfile
    rng = np.random.default_rng(seed)
    root.mkdir(parents=True, exist_ok=True)
    for i in range(n_files):
        x = O.synth_wav(rng, int(seconds * 44100), 44100)
        wavfile.write(root / f"clip{i}.wav", 44100, np.round(x * 32767).astype(np.int16))


INI = """[audio]
sampling_rate = 44100
hop_length = 128
segment_length = 1024

[dataset]
datapath = {data}
test_dataset = test_audio
generate_test = True
check_audio = True
check_dataset = True
workspace =
run_number = 0
total_frames =

[VAE]
latent_dim = 64
n_units = 256
kl_beta = 0.0001
device = cuda:0
{vae}
[training]
learning_rate = 0.0001
batch_size = 256
loss_reduction = mean
{training}

[notes]
additional_notes =

[extra]
normalize_examples = False
example_length = 10
plot_model = False
description = unit-test
start =
end =
time_elapsed =
"""


def _train(tmp, which, extra_training, extra_vae):
    from rawaudiovae_kelsey_b200 import trainer
    data = tmp / "data"
    _write_wavs(data / "audio", 3, 1.5, 1)
    _write_wavs(data / "test_audio", 1, 0.5, 2)
    ini = tmp / "t.ini"
    ini.write_text(INI.format(data=data, vae=extra_vae, training=extra_training))
    torch.manual_seed(0)
    random.seed(0)
    fn = trainer.run_epoch_trainer if which == "epoch" else trainer.run_stream_trainer
    assert fn(["--config", str(ini)]) in (0, None)
    return next((data / "unit-test").glob("run-*")), ini, data


@pytest.mark.parametrize("which", ["epoch", "stream"])
def test_trainer_logs_the_applied_schedule(which, dev, tmp_path):
    """A scheduled run logs the learning rate each step applies, over the run's own step count T, and KL Beta; a run
    with the default keys writes the tags it always wrote."""
    import configparser
    from rawaudiovae_kelsey_b200 import audio_io
    from rawaudiovae_kelsey_b200.dataset import AudioDataset, ToTensor
    from rawaudiovae_kelsey_b200.trainer import _epoch_trainer_steps, _schedule, _stream_trainer_steps
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    extra = ("epochs = 2\nsave_best_model_after = 1\ncheckpoint_interval = 2\nlog_interval = 4" if which == "epoch"
             else "epochs = 1\ntotal_num_frames = 2560\ncheckpoint_interval = 4\nlog_interval = 4")
    run, ini, data = _train(tmp_path / "a", which,
                            extra + "\nlr_schedule = cosine\nlr_warmup_steps = 2\nlr_min = 1e-6",
                            "kl_anneal = linear\nkl_anneal_steps = 5\n")
    base, _, _ = _train(tmp_path / "b", which, extra, "")
    sc, sb = _scalars(run), _scalars(base)
    cfg = configparser.ConfigParser()
    cfg.read(ini)
    if which == "epoch":
        chunks = [audio_io.load_mono(f, 44100)[0] for f in sorted((data / "audio").glob("*.wav"))]
        n_frames = len(AudioDataset(np.concatenate(chunks, axis=0), segment_length=1024, sampling_rate=44100,
                                    hop_size=128, transform=ToTensor()))
        T = _epoch_trainer_steps(cfg, n_frames)
    else:
        T = _stream_trainer_steps(cfg)
    sched = _schedule(cfg, T)
    lr0 = cfg["training"].getfloat("learning_rate")
    kb = cfg["VAE"].getfloat("kl_beta")
    assert sched.lr_schedule == "cosine" and sorted(sc["Learning Rate"]) == list(range(T))
    for k, v in sc["Learning Rate"].items():
        assert v == np.float32(sched.lr_at(k, lr0)), k
    assert sorted(sc["KL Beta"]) == list(range(T))
    for k, v in sc["KL Beta"].items():
        assert v == np.float32(sched.beta_at(k, kb)), k
    assert "KL Beta" not in sb
    assert set(sc) - set(sb) == {"KL Beta"}
    for k, v in sb["Learning Rate"].items():
        assert v == np.float32(lr0)
