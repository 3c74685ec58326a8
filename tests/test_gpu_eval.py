"""Held-out evaluation on the GPU: the per-frame loss kernel (rvae_frame_loss) against fp64, evaluate_audio against
the oracle and against loss_function, its independence of batch_size and of the training state, and the trainers'
[training] test_loss."""
import configparser
import random

import numpy as np
import pytest
import torch

from oracle import rawvae_oracle as O

pytestmark = pytest.mark.gpu

TOL = {"bf16": 2e-2, "fp32": 1e-4}
TAGS = {"Loss/test", "Loss/test_reconstruction", "Loss/test_kl"}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def maxrel(a, b):
    """max over frames of |a - b|, relative to the largest |b|: every frame, not a norm in which a few bad frames hide."""
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def make(dims, precision, dev, seed=0):
    from rawaudiovae_kelsey_b200.model import VAE
    p64 = {k: v.double() for k, v in O.init_params(*dims, seed=seed).items()}
    m = VAE(*dims, precision=precision)
    m.load_state_dict({k: v.float() for k, v in p64.items()})
    return m.to(dev), p64


def frames_of(audio32: np.ndarray, n: int, S: int, hop: int, first: int, rows: int) -> np.ndarray:
    """float64 [rows, S]: frame f = audio[(first + f) * hop + s], zeros at and beyond n."""
    a = np.zeros((first + rows) * hop + S, dtype=np.float64)
    a[:n] = audio32[:n]
    idx = (first + np.arange(rows))[:, None] * hop + np.arange(S)[None, :]
    return a[idx]


# ------------------------------------------------------------------------------------------------ 1. kernel vs fp64
CASES = [  # (S, L, hop, rows, first_frame, dtype)
    (1024, 256, 1024, 16384, 0, "f32"), (1024, 256, 256, 3000, 5, "i16"), (1024, 256, 1024, 700, 2, "i16"),
    (1000, 16, 200, 2000, 3, "f32"), (1000, 16, 1000, 513, 0, "i16"),
    (250, 3, 125, 1500, 1, "f32"), (250, 3, 250, 777, 0, "i16"),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "S{}-L{}-hop{}-rows{}-{}".format(c[0], c[1], c[2], c[3], c[5]))
def test_frame_loss_kernel_against_fp64(case, dev):
    from rawaudiovae_kelsey_b200 import ops
    S, L, hop, rows, first, kind = case
    ld_x, ld_l = -(-S // 64) * 64 + 64, -(-L // 64) * 64     # padded row pitches, wider than S / L
    g = torch.Generator().manual_seed(S + L + hop)
    n = (first + rows - 1) * hop + S // 2 + 3                  # the last frame runs past the end of the audio
    if kind == "f32":
        a = (torch.rand(n, generator=g) * 2 - 1).numpy().astype(np.float32)
        audio = torch.from_numpy(a).to(dev)
    else:
        pcm = torch.randint(-32768, 32768, (n,), generator=g, dtype=torch.int32).to(torch.int16)
        a = (pcm.float() / 32768.0).numpy()
        audio = pcm.to(dev)
    x = frames_of(a, n, S, hop, first, rows)
    xb = torch.full((rows, ld_x), float("nan"))                # padding columns must never be read
    xb[:, :S] = torch.from_numpy(x).float() + 0.05 * torch.randn(rows, S, generator=g)
    mb = torch.full((rows, ld_l), float("nan"))
    lb = torch.full((rows, ld_l), float("nan"))
    mb[:, :L] = torch.randn(rows, L, generator=g)
    lb[:, :L] = torch.randn(rows, L, generator=g) * 2
    xd, md, ld = xb.to(dev), mb.to(dev), lb.to(dev)
    rec, kl = ops.frame_loss(xd[:, :S], md[:, :L], ld[:, :L], audio, first, hop)
    rec2, kl2 = ops.frame_loss(xd[:, :S], md[:, :L], ld[:, :L], audio, first, hop)
    torch.cuda.synchronize()
    assert torch.equal(rec, rec2) and torch.equal(kl, kl2)     # deterministic
    xh = xb[:, :S].double().numpy()
    mu, lv = mb[:, :L].double().numpy(), lb[:, :L].double().numpy()
    rec_ref = ((xh - x) ** 2).mean(1)
    terms = 1 + lv - mu ** 2 - np.exp(lv)
    kl_ref = -0.5 * terms.mean(1)
    kl_mag = 0.5 * (1 + np.abs(lv) + mu ** 2 + np.exp(lv)).mean(1)
    r, k = rec.double().cpu().numpy(), kl.double().cpu().numpy()
    assert np.all(np.abs(r - rec_ref) <= 1e-6 * rec_ref), float(np.max(np.abs(r - rec_ref) / rec_ref))
    assert np.all(np.abs(k - kl_ref) <= 1e-6 * kl_mag), float(np.max(np.abs(k - kl_ref) / kl_mag))


# ------------------------------------------------------------------------------------------------ 2. vs the oracle
SHAPES = [((1024, 256, 64), 128), ((1000, 300, 16), 200), ((250, 100, 3), 125)]


@pytest.mark.parametrize("sample", [True, False], ids=["sample", "mean"])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_evaluate_audio_against_oracle(shape, precision, sample, dev):
    from rawaudiovae_kelsey_b200 import inference as I
    from rawaudiovae_kelsey_b200 import ops
    (S, H, L), hop = shape
    tol = TOL[precision]
    beta = 0.5
    model, p64 = make((S, H, L), precision, dev)
    wav = O.synth_wav(np.random.default_rng(1), hop * 151 + 37).astype(np.float32)
    for framing in (hop, None):
        frames = O.audio_dataset_frames(wav, S, framing) if framing else O.test_dataset_frames(wav, S)
        N = frames.shape[0]
        ev = I.evaluate_audio(model, wav, beta, hop=framing, batch_size=50, sample=sample, seed=3)
        eps = ops.randn((N, L), 3, 0, device=dev).double().cpu() if sample else torch.zeros(N, L, dtype=torch.float64)
        act = O.forward(p64, torch.from_numpy(np.ascontiguousarray(frames)).double(), eps)
        rec_ref = ((act["x_hat"] - act["x"]) ** 2).mean(1)
        kl_ref = -0.5 * (1 + act["logvar"] - act["mu"] ** 2 - torch.exp(act["logvar"])).mean(1)
        loss_ref = float(O.loss_function(act["x_hat"], act["x"], act["mu"], act["logvar"], beta, S))
        assert ev.reconstruction.shape == ev.kl.shape == (N,)
        assert ev.reconstruction.dtype == ev.kl.dtype == torch.float32
        assert maxrel(ev.reconstruction, rec_ref) < tol and maxrel(ev.kl, kl_ref) < tol, framing
        assert abs(ev.loss - loss_ref) <= tol * abs(loss_ref), (framing, ev.loss, loss_ref)
        assert abs(ev.reconstruction_mean - float(rec_ref.mean())) <= tol * float(rec_ref.mean())
        assert abs(ev.kl_mean - float(kl_ref.mean())) <= tol * abs(float(kl_ref.mean()))


# ------------------------------------------------------------------------------------------------ 3. vs loss_function
@pytest.mark.parametrize("shape", SHAPES[:2], ids=lambda s: "x".join(map(str, s[0])))
def test_loss_equals_loss_function_in_fp32_mode(shape, dev):
    from rawaudiovae_kelsey_b200 import inference as I
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import loss_function
    (S, H, L), hop = shape
    model, _ = make((S, H, L), "fp32", dev)
    wav = O.synth_wav(np.random.default_rng(2), hop * 301 + 11).astype(np.float32)
    x = torch.from_numpy(np.ascontiguousarray(O.audio_dataset_frames(wav, S, hop))).float().to(dev)
    N = x.shape[0]
    E = ops.randn((N, L), 0, 0, device=dev)
    counter = model._eps_counter
    ev = I.evaluate_audio(model, wav, 0.25, hop=hop, batch_size=N, seed=0)
    assert model._eps_counter == counter
    with torch.no_grad():
        xh, mu, lv = model(x, eps=E)
        ref = float(loss_function(xh, x, mu, lv, 0.25, S))
    assert abs(ev.loss - ref) <= 1e-6 * abs(ref), (ev.loss, ref)


# ------------------------------------------------------------------------------------------------ 4. batch_size
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_results_do_not_depend_on_batch_size(shape, dev):
    from rawaudiovae_kelsey_b200 import inference as I
    from rawaudiovae_kelsey_b200 import ops
    (S, H, L), hop = shape
    model, _ = make((S, H, L), "fp32", dev)
    wav = O.synth_wav(np.random.default_rng(4), hop * 211 + 5).astype(np.float32)
    N = I.frame_count(len(wav), S, hop)
    one = I.evaluate_audio(model, wav, 0.5, hop=hop, batch_size=N, seed=9)
    bs = N // 3 + 1
    split = I.evaluate_audio(model, wav, 0.5, hop=hop, batch_size=bs, seed=9)
    # the noise evaluate_audio draws: batch [lo, hi) is elements [lo L, hi L) of one Philox tensor, bit for bit
    full = ops.randn((N, L), 9, 0, device=dev)
    for lo in range(0, N, bs):
        hi = min(N, lo + bs)
        assert torch.equal(ops.randn((hi - lo, L), 9, 0, device=dev, elem_base=lo * L), full[lo:hi])
    for a, b in ((split.reconstruction, one.reconstruction), (split.kl, one.kl)):
        assert torch.allclose(a, b, rtol=1e-6, atol=1e-6 * float(b.abs().max()))
    print("batch-size independence bitwise:", torch.equal(split.reconstruction, one.reconstruction)
          and torch.equal(split.kl, one.kl))
    assert abs(split.loss - one.loss) <= 1e-6 * abs(one.loss)


# ------------------------------------------------------------------------------------------------ 5. side effects
def _state(model, opt):
    f = model._flat
    return [t.clone() for t in (f.params, f.grads, f.exp_avg, f.exp_avg_sq, f.step, f.shadow_hi)]


def test_no_side_effects_on_a_graph_prefetch_training_run(dev):
    """evaluate_audio between the steps of a FusedTrainStep(graph=True) run with next_data prefetch - so also between
    a step and the step that consumes its prefetched batch - changes no training state and no result."""
    from rawaudiovae_kelsey_b200 import inference as I
    from rawaudiovae_kelsey_b200.model import FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, hop, B, n = 1024, 256, 64, 128, 256, 8
    rng = np.random.default_rng(5)
    audio = torch.from_numpy(O.synth_wav(rng, hop * (B * (n + 1)) + S).astype(np.float32)).to(dev)
    held_out = O.synth_wav(rng, S * 300 + 17).astype(np.float32)
    batches = [FrameBatch(audio, B, hop, S, first_frame=i * B) for i in range(n)]

    def run(evaluate):
        model, _ = make((S, H, L), "bf16", dev)
        model.eps_seed = 7
        opt = Adam(model.parameters(), lr=1e-3)
        step = FusedTrainStep(model, opt, kl_beta=0.01, graph=True)
        losses, evals, inputs = [], [], []
        for i, b in enumerate(batches):
            losses.append(step(b, next_data=batches[i + 1] if i + 1 < n else None).clone())
            # the input set this step consumed: from step 1 on, the batch and noise prefetched by the step before,
            # with an evaluation in between (x as the converted sample span, read in place)
            cur = model._plan_for(B)
            assert cur.pitch == hop
            span = cur.activation("x")[0].reshape(-1)[:(B - 1) * hop + S]
            inputs.append((span.clone(), cur.latent("eps").clone()))
            if evaluate:
                plan = step._pf[0] if getattr(step, "_pf", None) else None
                pending = plan.prefetched_batch() if plan is not None else 0
                before, counter = _state(model, opt), model._eps_counter
                for bs in (B, 100):     # the training plan's batch size, and a smaller one with a ragged last batch
                    evals.append(I.evaluate_audio(model, held_out, 0.01, batch_size=bs, seed=0).loss)
                torch.cuda.synchronize()
                after = _state(model, opt)
                assert all(torch.equal(u, v) for u, v in zip(before, after)), i
                assert model._eps_counter == counter
                if plan is not None:
                    assert plan.prefetched_batch() == pending
        torch.cuda.synchronize()
        assert step.stats["replays"] > 0
        return torch.stack(losses), _state(model, opt), evals, inputs

    base, with_eval, again = run(False), run(True), run(False)
    for i, ((xa, ea), (xb, eb)) in enumerate(zip(with_eval[3], base[3])):
        assert torch.equal(xa, xb) and torch.equal(ea, eb), i
    assert all(abs(a - b) <= 1e-5 * abs(b) for a, b in zip(with_eval[2][::2], with_eval[2][1::2]))
    deterministic = torch.equal(base[0], again[0]) and all(torch.equal(u, v) for u, v in zip(base[1], again[1]))
    if deterministic:
        assert torch.equal(with_eval[0], base[0])
        assert all(torch.equal(u, v) for u, v in zip(with_eval[1], base[1]))
    # (split-K weight gradients and bias-gradient atomics reduce in no fixed order: two runs may differ in the last bits)
    assert torch.allclose(with_eval[0], base[0], rtol=1e-4, atol=0)
    assert rel(with_eval[1][0], base[1][0]) < 1e-3
    assert torch.equal(with_eval[1][4], base[1][4])        # step counter
    print("training run bitwise reproducible:", deterministic)


# ------------------------------------------------------------------------------------------------ 6. trainers
def _same_run(a, b):
    """Bitwise equal checkpoints and test_reconst_*.wav files."""
    for c in sorted((a / "model" / "checkpoints").glob("ckpt_*")):
        sa = torch.load(c, map_location="cpu", weights_only=False)["state_dict"]
        sb = torch.load(b / "model" / "checkpoints" / c.name, map_location="cpu", weights_only=False)["state_dict"]
        if not all(torch.equal(v, sb[k]) for k, v in sa.items()):
            return False
    return all((a / "audio_logs" / w.name).read_bytes() == (b / "audio_logs" / w.name).read_bytes()
               for w in (b / "audio_logs").glob("test_reconst_*.wav"))


def _scalars(run):
    from tensorboard.backend.event_processing.event_file_loader import LegacyEventFileLoader
    out = {}
    for f in sorted((run / "logs").glob("events.out.tfevents.*")):
        for ev in LegacyEventFileLoader(str(f)).Load():
            for v in ev.summary.value:
                if v.HasField("simple_value"):
                    out.setdefault(v.tag, {})[ev.step] = v.simple_value
                else:
                    out.setdefault(v.tag, {})
    return out


def _train(tmp, which, dims, hop, batch, extra, test_loss):
    from test_gpu_parity import _trainer_ini
    from test_gpu_param_histograms import _corpus
    from rawaudiovae_kelsey_b200 import trainer
    data = _corpus(tmp)
    ini = tmp / "t.ini"
    _trainer_ini(ini, data, batch=batch, extra_training=extra + ("\ntest_loss = True" if test_loss else ""))
    S, H, L = dims
    text = ini.read_text()
    for a, b in (("hop_length = 128", f"hop_length = {hop}"), ("segment_length = 1024", f"segment_length = {S}"),
                 ("latent_dim = 64", f"latent_dim = {L}"), ("n_units = 256", f"n_units = {H}")):
        text = text.replace(a, b)
    ini.write_text(text)
    torch.manual_seed(0)
    random.seed(0)   # the stream's file order (IterableAudioDataset.shuffled_data_list: random.sample)
    fn = trainer.run_epoch_trainer if which == "epoch" else trainer.run_stream_trainer
    assert fn(["--config", str(ini)]) in (0, None)
    return next((data / "unit-test").glob("run-*"))


TRAINERS = [
    ("epoch", (1024, 256, 64), 128, 512, "epochs = 3\nsave_best_model_after = 1\ncheckpoint_interval = 1"),
    ("epoch", (1000, 300, 16), 200, 200, "epochs = 3\nsave_best_model_after = 0\ncheckpoint_interval = 1"),
    ("stream", (1024, 256, 64), 128, 256, "epochs = 1\ntotal_num_frames = 2560\ncheckpoint_interval = 4\n"
                                           "log_interval = 3"),
]


@pytest.mark.parametrize("cfg", TRAINERS, ids=lambda c: "{}-{}".format(c[0], "x".join(map(str, c[1]))))
def test_trainer_logs_test_loss_and_keeps_the_best_model(cfg, dev, tmp_path):
    from rawaudiovae_kelsey_b200 import audio_io
    from rawaudiovae_kelsey_b200 import inference as I
    from rawaudiovae_kelsey_b200.model import VAE
    which, dims, hop, batch, extra = cfg
    on = _train(tmp_path / "on", which, dims, hop, batch, extra, True)
    off = _train(tmp_path / "off", which, dims, hop, batch, extra, False)
    off2 = _train(tmp_path / "off2", which, dims, hop, batch, extra, False)
    s_on, s_off = _scalars(on), _scalars(off)
    assert set(s_on) - set(s_off) == TAGS and set(s_off) <= set(s_on)
    # evaluation changes no training step: the per-batch losses agree (to the run-to-run spread of split-K
    # reductions, bitwise when two runs without test_loss are bitwise equal)
    steps = sorted(s_off["Loss/Batch"])
    assert steps and sorted(s_on["Loss/Batch"]) == steps
    a = torch.tensor([s_on["Loss/Batch"][k] for k in steps])
    b = torch.tensor([s_off["Loss/Batch"][k] for k in steps])
    assert torch.allclose(a, b, rtol=1e-4, atol=0)
    reproducible = _same_run(off, off2)
    if reproducible:
        assert _same_run(on, off) and torch.equal(a, b)
    print("trainer runs bitwise reproducible:", reproducible)
    ckpts = sorted((on / "model" / "checkpoints").glob("ckpt_*"))
    key = "epoch" if which == "epoch" else "batch_id"
    test_audio = audio_io.load_mono(next((on.parent.parent / "test_audio").glob("*.wav")), 44100)[0]
    losses = {}
    for c in ckpts:
        st = torch.load(c, map_location="cpu", weights_only=False)
        step_id = st[key]
        for tag in TAGS:
            assert step_id in s_on[tag], (tag, step_id, sorted(s_on[tag]))
        m = VAE(*dims).to(dev)
        m.load_state_dict(st["state_dict"])
        ev = I.evaluate_audio(m, test_audio, 0.0001, batch_size=batch, seed=0)
        for tag, v in (("Loss/test", ev.loss), ("Loss/test_reconstruction", ev.reconstruction_mean),
                       ("Loss/test_kl", ev.kl_mean)):
            assert abs(s_on[tag][step_id] - v) <= 1e-5 * abs(v), (tag, step_id, s_on[tag][step_id], v)
        losses[c.name] = (ev.loss, st)
        # the same run without test_loss: the same checkpoints and test audio, up to the run-to-run spread of training
        st_off = torch.load(off / "model" / "checkpoints" / c.name, map_location="cpu", weights_only=False)
        for k, v in st["state_dict"].items():
            assert rel(v, st_off["state_dict"][k]) < 1e-3, (c.name, k)
    assert len(ckpts) >= 2 and all(len(s_on[t]) == len(ckpts) for t in TAGS)
    wavs_on = sorted(p.name for p in (on / "audio_logs").glob("test_reconst_*.wav"))
    assert wavs_on == sorted(p.name for p in (off / "audio_logs").glob("test_reconst_*.wav")) and wavs_on
    for name in wavs_on:
        a = audio_io.load_mono(on / "audio_logs" / name, 44100)[0]
        b = audio_io.load_mono(off / "audio_logs" / name, 44100)[0]
        assert a.shape == b.shape and rel(torch.from_numpy(a), torch.from_numpy(b)) < 2e-2, name
    # best_model.pt = the checkpoint with the lowest test loss (after save_best_model_after for train.py)
    after = int(extra.split("save_best_model_after = ")[1].split("\n")[0]) if "save_best" in extra else -1
    eligible = {n: v for n, v in losses.items() if v[1][key] > after}
    best_name = min(eligible, key=lambda n: eligible[n][0])
    best = torch.load(on / "model" / "best_model.pt", map_location="cpu", weights_only=False)
    for k, v in best.state_dict().items():
        assert torch.equal(v, eligible[best_name][1]["state_dict"][k]), (best_name, k)
    cfg_out = configparser.ConfigParser(allow_no_value=True)
    cfg_out.read(on / "config.ini")
    best_key = "best_epoch" if which == "epoch" else "best_model"
    assert int(cfg_out["training"][best_key]) == eligible[best_name][1][key] or \
        (which == "stream" and best_name == ckpts[-1].name)
    assert abs(float(cfg_out["training"]["best_test_loss"]) - eligible[best_name][0]) <= 1e-5 * eligible[best_name][0]
