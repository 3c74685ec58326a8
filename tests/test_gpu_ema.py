"""Exponential moving average of the weights on the GPU: the standalone update against torch's AveragedModel, the EMA
inside the fused training step (eager, graph + prefetch, clipping, a cosine schedule, deterministic mode), decay
changes between replays, inference on ema.module, the state_dict round trip, two data-parallel ranks and the
trainers' checkpoints.

The reference is torch itself: AveragedModel(m, multi_avg_fn=get_ema_multi_avg_fn(decay)) with update_parameters
called on snapshots of the parameters after every step, on the same GPU. Both compute torch's two-branch lerp in fp32;
how nvcc contracts torch's lerp kernel into FMAs is not pinned down, so the comparison allows 1 ulp (equal_to_ulp)."""
import math
import os
import random
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn

from oracle import rawvae_oracle as O

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
DEFAULT = (1024, 2048, 256)           # default.ini
PADDED = (1000, 300, 16)              # padded to (1024, 320, 64) inside the plan
SMALL = (1024, 256, 64)
STATE = ("params", "exp_avg", "exp_avg_sq", "step")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def make(dims, precision, dev, seed=0):
    from rawaudiovae_kelsey_b200.model import VAE
    torch.manual_seed(seed)
    m = VAE(*dims, precision=precision)
    m.load_state_dict({k: v.float() for k, v in O.init_params(*dims, seed=seed).items()})
    return m.to(dev)


def true_mask(flat) -> torch.Tensor:
    m = torch.zeros_like(flat.params)
    for name in flat.geometry:
        flat.view(m, name).fill_(1.0)
    return m


class _Flat(torch.nn.Module):
    """One parameter holding a flat buffer: what AveragedModel averages in the reference."""

    def __init__(self, t):
        super().__init__()
        self.w = torch.nn.Parameter(t.detach().clone(), requires_grad=False)


class TorchEma:
    """torch's EMA of a sequence of flat parameter snapshots."""

    def __init__(self, like, decay):
        self.src = _Flat(like)
        self.avg = AveragedModel(self.src, multi_avg_fn=get_ema_multi_avg_fn(decay))

    def update(self, p):
        self.src.w.data.copy_(p)
        self.avg.update_parameters(self.src)

    @property
    def value(self):
        return self.avg.module.w.data


def _ordered(t):
    i = t.view(torch.int32).long()
    return torch.where(i < 0, -(i & 0x7FFFFFFF), i)


def equal_to_ulp(got, want, what=""):
    """Element for element equal, NaN where torch has NaN, infinities equal, finite values within 1 ulp."""
    assert got.shape == want.shape, what
    nan_g, nan_w = torch.isnan(got), torch.isnan(want)
    assert torch.equal(nan_g, nan_w), f"{what}: NaN positions differ"
    ok = ~nan_w
    g, w = got[ok], want[ok]
    inf = torch.isinf(w) | torch.isinf(g)
    assert torch.equal(g[inf], w[inf]), f"{what}: infinities differ"
    d = (_ordered(g[~inf]) - _ordered(w[~inf])).abs()
    if d.numel():
        assert int(d.max()) <= 1, f"{what}: {int(d.max())} ulp"


# ------------------------------------------------------------------------------------------------ the standalone update
@pytest.mark.parametrize("decay", [0.0, 0.5, 0.999, 1.0])
@pytest.mark.parametrize("dims", [DEFAULT, PADDED], ids=["default", "padded"])
def test_ema_update_matches_averaged_model(dims, decay, dev):
    from rawaudiovae_kelsey_b200 import ops
    model = make(dims, "bf16", dev)
    flat = model._ensure_flat()
    mask = true_mask(flat)
    gen = torch.Generator(device=dev).manual_seed(5)
    e = torch.randn(flat.total, generator=gen, device=dev) * mask
    decay_dev = torch.full((), decay, dtype=torch.float64, device=dev)
    count = torch.zeros((), dtype=torch.int64, device=dev)
    ref = TorchEma(e, decay)
    for k in range(5):
        p = torch.randn(flat.total, generator=gen, device=dev) * mask
        if k == 3:   # non-finite parameters propagate as in torch
            idx = mask.nonzero().flatten()
            p[idx[7]], p[idx[-3]], p[idx[len(idx) // 2]] = math.inf, -math.inf, math.nan
        ops.ema_update(e, p, decay_dev, count)
        ref.update(p)
        torch.cuda.synchronize()
        if k == 0:
            assert torch.equal(e, p), "the first update copies"
        equal_to_ulp(e, ref.value, f"update {k}")
        assert not bool(e[mask == 0].any()), "the padding stays 0"
    assert int(count) == 5 == int(ref.avg.n_averaged)


def test_ema_update_odd_length_and_argument_checks(dev):
    from rawaudiovae_kelsey_b200 import _lib, ops
    n = 4 * 148 * 256 * 4 + 7         # more than one grid pass, and a tail that is not a multiple of 4
    gen = torch.Generator(device=dev).manual_seed(1)
    e, decay_dev = torch.randn(n, generator=gen, device=dev), torch.full((), 0.9, dtype=torch.float64, device=dev)
    count = torch.ones((), dtype=torch.int64, device=dev)
    ref = TorchEma(e, 0.9)
    ref.avg.n_averaged.fill_(1)
    p = torch.randn(n, generator=gen, device=dev)
    ops.ema_update(e, p, decay_dev, count)
    ref.update(p)
    equal_to_ulp(e, ref.value, "odd length")
    assert int(count) == 2
    with pytest.raises(_lib.RvaeError):
        ops.ema_update(e[1:], p[1:], decay_dev, count)          # 4-byte offset: not 16-byte aligned


# ------------------------------------------------------------------------------------------------ inside the fused step
def _frames(dims, B, n, dev, hop=256, seed=3):
    from rawaudiovae_kelsey_b200.model import FrameBatch
    S = dims[0]
    wav = O.synth_wav(np.random.default_rng(seed), hop * (n * B + 20) + S).astype(np.float32)
    audio = torch.from_numpy(wav).to(dev)
    return [FrameBatch(audio, B, hop, S, first_frame=i * B) for i in range(n)]


def _train(dims, precision, dev, *, ema_decay=None, graph=True, prefetch=True, n=20, B=256, **kw):
    """n steps of FusedTrainStep; returns (state, ring, EMA, per-step parameter snapshots, step, eager launch count)."""
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.ema import ExponentialMovingAverage
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    model = make(dims, precision, dev)
    model.eps_seed = 11
    opt = Adam(model.parameters(), lr=1e-3)
    ema = ExponentialMovingAverage(model, ema_decay) if ema_decay is not None else None
    step = FusedTrainStep(model, opt, kl_beta=0.5, graph=graph, ema=ema, **kw)
    batches = _frames(dims, B, n, dev)
    snaps, launches = [], []
    for i, b in enumerate(batches):
        nxt = batches[i + 1] if prefetch and i + 1 < n else None
        l0 = ops.launch_count(dev)
        eager = step.stats["eager"]
        step(b, next_data=nxt)
        if step.stats["eager"] > eager:
            launches.append(ops.launch_count(dev) - l0)
        snaps.append(model._flat.params.clone())
    torch.cuda.synchronize()
    state = {k: getattr(model._flat, k).clone() for k in STATE}
    return state, step.ring.clone(), ema, snaps, step, launches


def _check_ema(ema, snaps, decay, what):
    ref = TorchEma(snaps[0], decay)
    for p in snaps:
        ref.update(p)
    equal_to_ulp(ema.target(), ref.value, what)
    assert int(ema.n_averaged) == len(snaps)


@pytest.mark.parametrize("mode", ["default", "deterministic"])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("dims", [DEFAULT, PADDED], ids=["default", "padded"])
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph-prefetch"])
def test_fused_step_ema(graph, dims, precision, mode, dev):
    """The EMA follows torch's on the step's own parameters, the padding stays 0, and an eager step launches as many
    kernels as without the EMA. In deterministic mode the run is the run without the EMA bit for bit: parameters,
    moments, step counter and loss ring (the default step reduces split-K gradients with atomics, so two of its runs
    drift apart whether or not the EMA is on)."""
    kw = dict(graph=graph, prefetch=graph, deterministic=mode == "deterministic")
    s1, r1, ema, snaps, step, l1 = _train(dims, precision, dev, ema_decay=0.9, **kw)
    s0, r0, _, _, _, l0 = _train(dims, precision, dev, **kw)
    _check_ema(ema, snaps, 0.9, f"{precision} {graph} {mode}")
    assert not bool(ema.target()[true_mask(ema.module._flat) == 0].any())
    assert l1 == l0 and l1, (l1, l0)
    if graph:
        assert step.stats["replays"] >= 10
    assert torch.equal(s1["step"], s0["step"])
    if mode == "deterministic":
        for k in STATE:
            assert torch.equal(s1[k], s0[k]), f"{k} differs with the EMA on"
        assert torch.equal(r1, r0), "loss ring"


@pytest.mark.parametrize("case", ["clip-cosine", "deterministic", "deterministic-clip-cosine"])
@pytest.mark.parametrize("dims", [SMALL, PADDED], ids=["small", "padded"])
def test_ema_composes_with_clipping_schedules_and_deterministic_mode(case, dims, dev):
    from rawaudiovae_kelsey_b200.schedule import Schedule
    kw = {}
    if "clip" in case:
        kw.update(max_grad_norm=1e-3, schedule=Schedule(lr_schedule="cosine", warmup_steps=4, total_steps=20))
    if "deterministic" in case:
        kw.update(deterministic=True)
    s1, r1, ema, snaps, step, l1 = _train(dims, "bf16", dev, ema_decay=0.95, **kw)
    _check_ema(ema, snaps, 0.95, case)
    assert step.stats["replays"] >= 10
    if "deterministic" in case:
        s0, r0, _, _, _, l0 = _train(dims, "bf16", dev, **kw)
        for k in STATE:
            assert torch.equal(s1[k], s0[k]), f"{k} differs with the EMA on"
        assert torch.equal(r1, r0), "loss ring"
        s2, _, ema2, _, _, _ = _train(dims, "bf16", dev, ema_decay=0.95, **kw)
        assert torch.equal(ema.target(), ema2.target()), "two deterministic runs give different EMAs"
        assert torch.equal(s1["params"], s2["params"])


def test_decay_changes_reach_replays_and_the_ema_switches_on_mid_run(dev):
    from rawaudiovae_kelsey_b200.ema import ExponentialMovingAverage
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    model = make(SMALL, "bf16", dev)
    model.eps_seed = 2
    opt = Adam(model.parameters(), lr=1e-3)
    x = torch.from_numpy(O.synth_wav(np.random.default_rng(2), 1024 * 256).astype(np.float32)).to(dev)
    x = x.reshape(256, 1024)
    plain = FusedTrainStep(model, opt, kl_beta=0.5, graph=True)
    for _ in range(3):          # a resumed optimizer: the step counter is past 0 when the EMA starts
        plain(x)
    ema = ExponentialMovingAverage(model, decay=0.5)
    step = FusedTrainStep(model, opt, kl_beta=0.5, graph=True, ema=ema)
    step(x)
    torch.cuda.synchronize()
    assert torch.equal(ema.target(), model._flat.params), "the first update copies"
    assert int(ema.n_averaged) == 1 and int(model._flat.step) == 4
    ref = TorchEma(model._flat.params, 0.5)
    ref.update(model._flat.params)
    for _ in range(2):
        step(x)
        ref.update(model._flat.params)
    assert step.stats["captures"] == 1
    for decay in (0.9, 0.0, 1.0, 0.999):
        ema.decay = decay
        ref.avg.multi_avg_fn = get_ema_multi_avg_fn(decay)
        replays = step.stats["replays"]
        step(x)
        ref.update(model._flat.params)
        torch.cuda.synchronize()
        assert step.stats["replays"] == replays + 1 and step.stats["captures"] == 1
        equal_to_ulp(ema.target(), ref.value, f"decay {decay}")
    assert int(ema.n_averaged) == 7


@pytest.mark.parametrize("dims", [DEFAULT, PADDED], ids=["default", "padded"])
def test_module_inference_follows_the_ema_and_the_state_dict_round_trips(dims, dev):
    from rawaudiovae_kelsey_b200.ema import ExponentialMovingAverage
    from rawaudiovae_kelsey_b200.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    model = make(dims, "bf16", dev)
    ema = ExponentialMovingAverage(model, decay=0.8)
    step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-3), kl_beta=0.5, graph=True, ema=ema)
    x = torch.from_numpy(O.synth_wav(np.random.default_rng(4), dims[0] * 256).astype(np.float32)).to(dev)
    x = x.reshape(256, dims[0])
    eps = torch.randn(256, dims[2], generator=torch.Generator(device=dev).manual_seed(0), device=dev)
    prev = None
    for rounds in range(3):
        for _ in range(4):
            step(x)
        fresh = VAE(*dims).to(dev)
        fresh.load_state_dict(ema.state_dict())
        with torch.no_grad():
            mu, lv = ema.module.encode(x)
            xh = ema.module(x, eps=eps)[0]
            mu_f, lv_f = fresh.encode(x)
            xh_f = fresh(x, eps=eps)[0]
        assert torch.equal(mu, mu_f) and torch.equal(lv, lv_f) and torch.equal(xh, xh_f), rounds
        if prev is not None:
            assert not torch.equal(mu, prev), "ema.module did not follow the steps"
        prev = mu
    sd = ema.state_dict()
    assert list(sd) == list(VAE(*dims).state_dict())
    assert all(v.is_contiguous() for v in sd.values())
    ref = VAE(*dims)                        # the reference module structure, on the CPU
    ref.load_state_dict({k: v.cpu() for k, v in sd.items()})
    p64 = {k: v.double() for k, v in ref.state_dict().items()}
    assert set(p64) == set(O.init_params(*dims))
    n_avg = int(ema.n_averaged)
    other = ExponentialMovingAverage(make(dims, "bf16", dev, seed=1), decay=0.8)
    other.load_state_dict(sd, n_averaged=ema.n_averaged)
    assert int(other.n_averaged) == n_avg
    assert torch.equal(other.target(), ema.target())
    with torch.no_grad():
        assert torch.equal(other.module.encode(x)[0], prev)


def test_unfused_path_update(dev):
    """loss.backward(); optimizer.step(); ema.update() - the EMA of the parameters after each optimizer step."""
    from rawaudiovae_kelsey_b200.ema import ExponentialMovingAverage
    from rawaudiovae_kelsey_b200.model import loss_function
    from rawaudiovae_kelsey_b200.optim import Adam
    model = make(SMALL, "bf16", dev)
    opt = Adam(model.parameters(), lr=1e-3)
    ema = ExponentialMovingAverage(model, decay=0.7)
    ref = None
    x = torch.from_numpy(O.synth_wav(np.random.default_rng(6), 1024 * 128).astype(np.float32)).to(dev)
    x = x.reshape(128, 1024)
    for _ in range(4):
        opt.zero_grad()
        xh, mu, lv = model(x)
        loss_function(xh, x, mu, lv, 0.5, 1024).backward()
        opt.step()
        ema.update()
        p = model._flat.params
        if ref is None:
            ref = TorchEma(p, 0.7)
        ref.update(p)
    equal_to_ulp(ema.target(), ref.value, "unfused")
    assert int(ema.n_averaged) == 4


# ------------------------------------------------------------------------------------------------ data parallel
def _free_port():
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    port = sk.getsockname()[1]
    sk.close()
    return port


def _dp_worker(rank, world, port, ret):
    sys.path.insert(0, str(ROOT))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from rawaudiovae_kelsey_b200 import dist as rdist
    from rawaudiovae_kelsey_b200.dataset import shard_bounds
    from rawaudiovae_kelsey_b200.ema import ExponentialMovingAverage
    from rawaudiovae_kelsey_b200.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    _, _, local = rdist.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    S, H, L, B, n = 1024, 256, 64, 1000, 6
    gen = torch.Generator().manual_seed(1)
    x = (torch.rand(B, S, generator=gen) * 2 - 1).to(dev)

    def build():
        torch.manual_seed(0)
        m = VAE(S, H, L).to(dev)
        m.eps_seed = 123
        return m, Adam(m.parameters(), lr=1e-3), ExponentialMovingAverage(m, decay=0.9)

    m_dp, o_dp, e_dp = build()
    m_1, o_1, e_1 = build()
    step_dp = rdist.DataParallelTrainStep(m_dp, o_dp, 0.5, global_batch=B, graph=True, ema=e_dp)
    step_1 = FusedTrainStep(m_1, o_1, 0.5, graph=True, ema=e_1)
    lo, hi = shard_bounds(B, rank, world)
    for _ in range(n):
        step_dp(x[lo:hi].contiguous())
        step_1(x)
    torch.cuda.synchronize()
    a, b = e_dp.target().double(), e_1.target().double()
    de = float((a - b).norm() / b.norm())
    ref = e_dp.target().clone()
    dist.broadcast(ref, src=0)
    same = bool(torch.equal(ref, e_dp.target())) and int(e_dp.n_averaged) == n
    ret.put((rank, same, de, step_dp.stats["replays"]))
    dist.barrier()
    dist.destroy_process_group()


def test_data_parallel_ema_is_identical_on_every_rank(dev):
    """2 ranks, graph=True: the averages are bitwise equal across ranks and match the single process on the whole
    batch within tools/dp_check.py's weight tolerance (4e-3 relative)."""
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
    for rank, same, de, rep in sorted(out):
        assert rep > 0 and same, rank
        assert de < 4e-3, (rank, de)


# ------------------------------------------------------------------------------------------------ trainers
def _scalar_tags(run):
    from tensorboard.backend.event_processing.event_file_loader import LegacyEventFileLoader
    tags = set()
    for f in sorted((run / "logs").glob("events.out.tfevents.*")):
        for ev in LegacyEventFileLoader(str(f)).Load():
            tags.update(v.tag for v in ev.summary.value)
    return tags


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


def _run_trainer(tmp, which, extra_training):
    from rawaudiovae_kelsey_b200 import trainer
    data = tmp / "data"
    _write_wavs(data / "audio", 3, 1.5, 1)
    _write_wavs(data / "test_audio", 1, 0.5, 2)
    ini = tmp / "t.ini"
    ini.write_text(INI.format(data=data, training=extra_training))
    torch.manual_seed(0)
    random.seed(0)
    fn = trainer.run_epoch_trainer if which == "epoch" else trainer.run_stream_trainer
    assert fn(["--config", str(ini)]) in (0, None)
    return next((data / "unit-test").glob("run-*"))


@pytest.mark.parametrize("which", ["epoch", "stream"])
def test_trainer_saves_the_ema(which, dev, tmp_path):
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    extra = ("epochs = 2\nsave_best_model_after = 0\ncheckpoint_interval = 1\nlog_interval = 4\ntest_loss = True"
             if which == "epoch" else
             "epochs = 1\ntotal_num_frames = 2560\ncheckpoint_interval = 4\nlog_interval = 4\ntest_loss = True")
    run_e = _run_trainer(tmp_path / "a", which, extra + "\nema_decay = 0.9")
    run_p = _run_trainer(tmp_path / "b", which, extra)
    ck_e = sorted((run_e / "model" / "checkpoints").glob("ckpt_*"))
    ck_p = sorted((run_p / "model" / "checkpoints").glob("ckpt_*"))
    assert ck_e and len(ck_e) == len(ck_p)
    plain_keys = set(torch.load(ck_p[-1], weights_only=False))
    assert "ema_state_dict" not in plain_keys and "ema_n_averaged" not in plain_keys
    last = torch.load(ck_e[-1], weights_only=False)
    assert set(last) == plain_keys | {"ema_state_dict", "ema_n_averaged"}
    assert last["ema_n_averaged"] > 0
    assert set(last["ema_state_dict"]) == set(last["state_dict"])
    assert any(not torch.equal(last["ema_state_dict"][k].cpu(), last["state_dict"][k].cpu())
               for k in last["state_dict"]), "the EMA equals the raw weights"
    lm = torch.load(run_e / "model" / "last_model.pt", weights_only=False)
    for k, v in lm.state_dict().items():
        assert torch.equal(v.cpu(), last["ema_state_dict"][k].cpu()), k      # last_model.pt holds the EMA
    assert (run_e / "model" / "best_model.pt").exists()
    best = torch.load(run_e / "model" / "best_model.pt", weights_only=False)
    raw = {k: v.cpu() for k, v in last["state_dict"].items()}
    assert any(not torch.equal(v.cpu(), raw[k]) for k, v in best.state_dict().items())
    assert _scalar_tags(run_e) == _scalar_tags(run_p)
