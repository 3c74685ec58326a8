"""Gradient-norm clipping inside the fused training step on the GPU: the norm reduction on crafted gradients, the
clipped Adam update step by step, graph + prefetch training against the fp64 oracle, the unfused torch path,
changes of the threshold between replays, the 2-rank data-parallel step and the trainers' Grad Norm tag."""
import math
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
DEFAULT = (1024, 2048, 256)           # default.ini
PADDED = (1000, 300, 16)              # padded to (1024, 320, 64) inside the plan


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


def ulp32(x: float) -> float:
    x = np.float32(abs(x))
    return float(np.nextafter(x, np.float32(np.inf)) - x)


def norm64(t: torch.Tensor) -> float:
    t = t.double()
    return math.sqrt(float((t * t).sum()))


def clip_coef(norm: float, max_norm: float) -> float:
    """The factor the step applies: min(1, max_norm / (norm + 1e-6)) in fp64, rounded to fp32 once."""
    return float(np.float32(min(1.0, max_norm / (norm + 1e-6))))


def true_mask(flat) -> torch.Tensor:
    """1 at the true parameters of the flat buffer, 0 at the padding of padded dims."""
    m = torch.zeros_like(flat.params)
    for name in flat.geometry:
        flat.view(m, name).fill_(1.0)
    return m


# ------------------------------------------------------------------------------------------------ the reduction
@pytest.mark.parametrize("dims", [DEFAULT, PADDED], ids=["default", "padded"])
def test_grad_norm_on_crafted_gradients(dims, dev):
    from rawaudiovae_kelsey_b200.engine import Plan
    model = make(dims, "bf16", dev)
    flat = model._ensure_flat()
    plan = Plan(flat, 256)
    mask = true_mask(flat)
    gen = torch.Generator(device=dev).manual_seed(7)

    def fill(scale):
        flat.grads.copy_(torch.randn(flat.total, generator=gen, device=dev) * scale * mask)

    for scale in (1.0, 1e-3, 1e4, 1e-30):
        fill(scale)
        want = norm64(flat.grads)
        outs = [plan.grad_norm().clone() for _ in range(3)]
        torch.cuda.synchronize()
        got = float(outs[0])
        assert got > 0.0, scale                                   # 1e-30 squared in fp64 does not underflow
        assert abs(got - want) <= ulp32(want), (scale, got, want)
        assert all(torch.equal(o, outs[0]) for o in outs[1:])     # bitwise repeatable
    # a non-finite element propagates, wherever it sits
    for bad, check in ((math.inf, math.isinf), (math.nan, math.isnan)):
        for pos in (0, flat.total // 2, flat.total - 1):
            fill(1.0)
            flat.grads[pos] = bad
            assert check(float(plan.grad_norm())), (bad, pos)


# ------------------------------------------------------------------------------------------------ the clipped update
def _host_adam(p0, m0, v0, g, t, lr):
    m = m0.double() + (1 - 0.9) * (g - m0.double())
    v = 0.999 * v0.double() + (1 - 0.999) * g * g
    return p0.double() - lr / (1 - 0.9 ** t) * m / (v.sqrt() / (1 - 0.999 ** t) ** 0.5 + 1e-8)


def _check_update(flat, p0, m0, v0, g_kept, t, lr, coef):
    """The tolerance of test_adam_applies_the_scheduled_lr: 1e-6 of the update plus half an ulp of the result."""
    p1 = flat.params.double()
    scale = float((p1 - p0.double()).abs().max())
    ulp = (torch.nextafter(flat.params.abs(), torch.tensor(float("inf"), device=flat.params.device))
           - flat.params.abs()).double()
    g = (g_kept * torch.tensor(coef, dtype=torch.float32, device=g_kept.device)).double()   # fp32 g * coef
    err = (p1 - _host_adam(p0, m0, v0, g, t, lr)).abs()
    assert bool((err <= 1e-6 * scale + 0.5 * ulp).all()), (t, float(err.max()), scale)


@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("max_norm", [1e-3, 1e6], ids=["binding", "not-binding"])
def test_clipped_step_updates_with_coef_times_g(max_norm, precision, graph, dev):
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    model = make((1024, 256, 64), precision, dev)
    model.eps_seed = 5
    opt = Adam(model.parameters(), lr=1e-3)
    step = FusedTrainStep(model, opt, kl_beta=0.5, keep_grads=True, graph=graph, max_grad_norm=max_norm)
    x = torch.from_numpy(O.synth_wav(np.random.default_rng(1), 1024 * 256).astype(np.float32)).to(dev)
    x = x.reshape(256, 1024)
    flat = model._flat
    for k in range(5):
        p0, m0, v0 = flat.params.clone(), flat.exp_avg.clone(), flat.exp_avg_sq.clone()
        step(x)
        torch.cuda.synchronize()
        g = flat.grads.clone()                     # the kept gradients: raw, unclipped
        n = norm64(g)
        got = float(step.grad_norm)
        assert abs(got - n) <= ulp32(n), (k, got, n)
        coef = clip_coef(n, max_norm)
        assert (coef < 1.0) == (max_norm == 1e-3), (k, n)
        _check_update(flat, p0, m0, v0, g.double(), k + 1, 1e-3, coef)
        if coef == 1.0:
            # no clipping: bit for bit the update of the plain fused Adam kernel on the same state and gradient
            p, m, v = p0.clone(), m0.clone(), v0.clone()
            st = torch.tensor(float(k), device=dev)
            ops.adam_step(p, g, m, v, st, 1e-3)
            torch.cuda.synchronize()
            assert torch.equal(p, flat.params) and torch.equal(m, flat.exp_avg) and torch.equal(v, flat.exp_avg_sq)
    if graph:
        assert step.stats["replays"] >= 3


# ------------------------------------------------------------------------------------------------ against the oracle
def _oracle_clipped_step(p64, state, x, eps, kl_beta, lr, max_norm, q=lambda t: t):
    """O.train_step with torch.nn.utils.clip_grad_norm_ (fp64) between backward and Adam."""
    act = O.forward(p64, x, eps, q)
    S = p64["fc1.weight"].shape[1]
    loss = O.loss_function(act["x_hat"], act["x"], act["mu"], act["logvar"], kl_beta, S)
    grads = {k: O.backward(p64, act, kl_beta, 1.0, q)[k] for k in O.PARAM_NAMES}   # (without the activation grads)
    norm = math.sqrt(sum(float((g * g).sum()) for g in grads.values()))
    coef = min(1.0, max_norm / (norm + 1e-6))
    O.adam_step(p64, {k: g * coef for k, g in grads.items()}, state, lr)
    return float(loss), norm


@pytest.mark.parametrize("dims, hop, precision", [((1024, 256, 64), 256, "bf16"), ((1024, 256, 64), 256, "fp32"),
                                                  (PADDED, 200, "bf16"), (PADDED, 200, "fp32")])
def test_graph_prefetch_training_matches_the_clipped_oracle(dims, hop, precision, dev):
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    S, L = dims[0], dims[2]
    B, n, max_norm = 256, 6, 1e-3
    wav = O.synth_wav(np.random.default_rng(3), hop * (n * B + 20) + S).astype(np.float32)
    audio = torch.from_numpy(wav).to(dev)
    batches = [FrameBatch(audio, B, hop, S, first_frame=i * B) for i in range(n)]
    model = make(dims, precision, dev)
    model.eps_seed = 11
    opt = Adam(model.parameters(), lr=1e-3)
    step = FusedTrainStep(model, opt, kl_beta=0.5, graph=True, max_grad_norm=max_norm)
    losses, norms, early = [], [], None
    for i, b in enumerate(batches):
        losses.append(step(b, next_data=batches[i + 1] if i + 1 < n else None).clone())
        norms.append(step.grad_norm.clone())
        if i == 2:
            early = {k: v.detach().clone() for k, v in model.state_dict().items()}
    torch.cuda.synchronize()
    assert step.stats["replays"] >= 1
    p64 = {k: v.double() for k, v in O.init_params(*dims, seed=0).items()}
    state = O.adam_init(p64)
    frames = torch.from_numpy(O.audio_dataset_frames(wav, S, hop)).double()
    ref, ref_norm, par_err = [], [], None
    for k in range(3):
        eps = ops.randn((B, L), 11, k, device=dev).double().cpu()
        loss, nrm = _oracle_clipped_step(p64, state, frames[k * B:(k + 1) * B], eps, 0.5, 1e-3, max_norm)
        ref.append(loss)
        ref_norm.append(nrm)
    par_err = max(rel(v, p64[name]) for name, v in early.items())
    assert min(ref_norm) > max_norm                       # clipping binds at every compared step
    loss_err = max(abs(float(losses[k]) - ref[k]) / abs(ref[k]) for k in range(3))
    norm_err = max(abs(float(norms[k]) - ref_norm[k]) / ref_norm[k] for k in range(3))
    assert loss_err <= TOL[precision], loss_err
    assert norm_err <= TOL[precision], norm_err
    assert par_err <= {"fp32": 1e-3, "bf16": TOL["bf16"]}[precision], par_err
    mask = true_mask(model._flat)
    for buf in ("params", "exp_avg", "exp_avg_sq"):
        assert not bool(getattr(model._flat, buf)[mask == 0].any()), buf     # the padding stays exactly zero
    assert all(math.isfinite(float(v)) for v in norms)


# ------------------------------------------------------------------------------------------------ against the unfused path
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_fused_clipped_step_matches_unfused_torch_clipping(precision, dev):
    from rawaudiovae_kelsey_b200.model import FusedTrainStep, loss_function
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, B, max_norm = 1024, 256, 64, 256, 1e-3
    gen = torch.Generator().manual_seed(1)
    x = (torch.rand(B, S, generator=gen) * 2 - 1).to(dev)
    eps = torch.randn(B, L, generator=gen).to(dev)

    def unfused():
        model = make((S, H, L), precision, dev)
        opt = Adam(model.parameters(), lr=1e-3)
        losses, norms = [], []
        for _ in range(3):
            opt.zero_grad()
            xh, mu, lv = model(x, eps=eps)
            loss = loss_function(xh, x, mu, lv, 0.5, S)
            loss.backward()
            norms.append(float(torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm)))
            opt.step()
            losses.append(float(loss))
        return model, losses, norms

    def fused():
        model = make((S, H, L), precision, dev)
        opt = Adam(model.parameters(), lr=1e-3)
        step = FusedTrainStep(model, opt, kl_beta=0.5, max_grad_norm=max_norm)
        losses, norms = [], []
        for _ in range(3):
            losses.append(float(step(x, eps=eps)))
            norms.append(float(step.grad_norm))
        return model, losses, norms

    mu_, lu, nu = unfused()
    mf, lf, nf = fused()
    assert min(nu) > max_norm
    for a, b in zip(lf, lu):
        assert abs(a - b) <= TOL[precision] * abs(b), (lf, lu)
    for a, b in zip(nf, nu):
        assert abs(a - b) <= TOL[precision] * abs(b), (nf, nu)
    for name, p in mu_.state_dict().items():
        assert rel(mf.state_dict()[name], p) <= {"fp32": 1e-3, "bf16": TOL["bf16"]}[precision], name


# ------------------------------------------------------------------------------------------------ host changes and replays
def test_threshold_changes_reach_replays_and_switching_off_restores_the_update(dev):
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    model = make((1024, 256, 64), "bf16", dev)
    model.eps_seed = 2
    opt = Adam(model.parameters(), lr=1e-3)
    step = FusedTrainStep(model, opt, kl_beta=0.5, keep_grads=True, graph=True, max_grad_norm=1e6)
    x = torch.from_numpy(O.synth_wav(np.random.default_rng(2), 1024 * 256).astype(np.float32)).to(dev)
    x = x.reshape(256, 1024)
    for _ in range(3):
        step(x)
    assert step.stats["captures"] == 1
    flat = model._flat
    for max_norm in (1e-3, 2e-3, math.inf):
        step.max_grad_norm = max_norm
        torch.cuda.synchronize()
        p0, m0, v0, t = flat.params.clone(), flat.exp_avg.clone(), flat.exp_avg_sq.clone(), int(flat.step)
        replays = step.stats["replays"]
        step(x)
        torch.cuda.synchronize()
        assert step.stats["replays"] == replays + 1 and step.stats["captures"] == 1
        g = flat.grads.clone()
        n = norm64(g)
        assert abs(float(step.grad_norm) - n) <= ulp32(n)
        _check_update(flat, p0, m0, v0, g.double(), t + 1, 1e-3, clip_coef(n, max_norm))
    # off: not served by the clipping graph, and the update of an unclipped step from the same state
    step.max_grad_norm = None
    snap = {k: getattr(flat, k).clone() for k in ("params", "exp_avg", "exp_avg_sq", "step")}
    replays = step.stats["replays"]
    step(x)
    torch.cuda.synchronize()
    assert step.stats["replays"] == replays and step.grad_norm is None
    got = {k: getattr(flat, k).clone() for k in ("params", "exp_avg", "exp_avg_sq", "step")}
    for k, v in snap.items():
        getattr(flat, k).copy_(v)
    flat.sync_shadow()
    plain = FusedTrainStep(model, opt, kl_beta=0.5, keep_grads=True)
    plain(x)
    torch.cuda.synchronize()
    assert norm64(flat.grads) > 2e-3                          # the thresholds above did bind
    # split-K reduction order makes two unclipped steps differ in the last bits: moments within 1e-4, the parameter
    # update (Adam amplifies near-zero gradients) within 1e-2; a clipped step's moments differ by far more
    assert torch.equal(flat.step, got["step"])
    assert rel(flat.exp_avg, got["exp_avg"]) <= 1e-4 and rel(flat.exp_avg_sq, got["exp_avg_sq"]) <= 1e-4
    assert rel(flat.params - snap["params"], got["params"] - snap["params"]) <= 1e-2


# ------------------------------------------------------------------------------------------------ data parallel
def _free_port():
    sk = socket.socket()
    sk.bind(("127.0.0.1", 0))
    port = sk.getsockname()[1]
    sk.close()
    return port


def _dp_worker(rank, world, port, ret):
    """One rank: the clipped DataParallelTrainStep on its shard and the clipped single-process FusedTrainStep on the
    whole batch, both graph=True with Philox noise, from identical weights."""
    sys.path.insert(0, str(ROOT))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from rawaudiovae_kelsey_b200 import dist as rdist
    from rawaudiovae_kelsey_b200.dataset import shard_bounds
    from rawaudiovae_kelsey_b200.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    _, _, local = rdist.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    S, H, L, B, n, max_norm = 1024, 256, 64, 1000, 6, 1e-3
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
                                          max_grad_norm=max_norm)
    step_1 = FusedTrainStep(m_1, o_1, 0.5, graph=True, max_grad_norm=max_norm)
    lo, hi = shard_bounds(B, rank, world)
    dl = dn = 0.0
    norms = []
    for _ in range(n):
        l_dp = step_dp(x[lo:hi].contiguous())
        l_1 = step_1(x)
        torch.cuda.synchronize()
        dl = max(dl, abs(float(l_dp) - float(l_1)) / float(l_1))
        dn = max(dn, abs(float(step_dp.grad_norm) - float(step_1.grad_norm)) / float(step_1.grad_norm))
        norms.append(step_dp.grad_norm.clone())
    norms = torch.stack(norms)
    dw = float((m_dp._flat.params.double() - m_1._flat.params.double()).norm() / m_1._flat.params.double().norm())
    ref, ref_n = m_dp._flat.params.clone(), norms.clone()
    if dist.is_initialized():
        dist.broadcast(ref, src=0)
        dist.broadcast(ref_n, src=0)
    same = bool(torch.equal(ref, m_dp._flat.params)) and bool(torch.equal(ref_n, norms))
    binding = bool((norms > max_norm).all())
    ret.put((rank, same, binding, dl, dn, dw, step_dp.stats["replays"]))
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()


def test_data_parallel_clipping_keeps_replicas_equal(dev):
    """2 ranks, graph=True, clipping binding: the replicas and their norm rings stay bitwise equal, and match the
    single process on the whole batch within tools/dp_check.py's tolerances (loss 1e-4, weights 4e-3 relative)."""
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
    for rank, same, binding, dl, dn, dw, rep in sorted(out):
        assert rep > 0 and same and binding, rank
        assert dl < 1e-4 and dn < 1e-4 and dw < 4e-3, (rank, dl, dn, dw)


# ------------------------------------------------------------------------------------------------ trainers
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


def _train(tmp, which, extra_training):
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
def test_trainer_logs_grad_norm(which, dev, tmp_path):
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    extra = ("epochs = 2\nsave_best_model_after = 1\ncheckpoint_interval = 2\nlog_interval = 4" if which == "epoch"
             else "epochs = 1\ntotal_num_frames = 2560\ncheckpoint_interval = 4\nlog_interval = 4")
    sc = _scalars(_train(tmp_path / "a", which, extra + "\nmax_grad_norm = 1.0"))
    sb = _scalars(_train(tmp_path / "b", which, extra))
    assert set(sc) - set(sb) == {"Grad Norm"} and set(sb) <= set(sc)
    assert sorted(sc["Grad Norm"]) == sorted(sc["Loss/Batch"])        # one norm per step, at the step id
    assert all(math.isfinite(v) and v > 0 for v in sc["Grad Norm"].values())
