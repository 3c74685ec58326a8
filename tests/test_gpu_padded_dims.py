"""A VAE whose segment_length / n_units / latent_dim are not multiples of 64, against the fp64 oracle.

(1000, 300, 16): S a multiple of 8 but not of 64, small L; frames at hop 200 are read in place (bf16 mode).
(250, 100, 3): S not a multiple of 8, L not a multiple of 4; frames at hop 125 are gathered."""
import copy

import numpy as np
import pytest
import torch

from oracle import rawvae_oracle as O

pytestmark = pytest.mark.gpu

SHAPES = [((1000, 300, 16), 200, 200), ((250, 100, 3), 125, 300)]   # (dims, hop, batch)
TOL = {"bf16": 2e-2, "fp32": 1e-4}


def check_histogram(fields, values, edges, what):
    """add_histogram_raw fields == TensorBoard's make_histogram of the values: limits, counts, min, max, num exactly."""
    from torch.utils.tensorboard.summary import make_histogram
    ref = make_histogram(np.asarray(values, dtype=np.float64), edges)
    assert list(fields["bucket_limits"]) == list(ref.bucket_limit), what
    assert list(fields["bucket_counts"]) == list(ref.bucket), what
    assert (fields["min"], fields["max"], fields["num"]) == (ref.min, ref.max, ref.num), what
    assert abs(fields["sum"] - ref.sum) <= 1e-12 * abs(ref.sum) + 1e-300, what
    assert abs(fields["sum_squares"] - ref.sum_squares) <= 1e-12 * ref.sum_squares, what


class RefVAE(torch.nn.Module):
    """The reference's module structure at given dims (rawvae/model.py:13-17), plain torch: what a checkpoint must
    load into."""

    def __init__(self, S, H, L):
        super().__init__()
        self.fc1, self.fc21, self.fc22 = torch.nn.Linear(S, H), torch.nn.Linear(H, L), torch.nn.Linear(H, L)
        self.fc3, self.fc4 = torch.nn.Linear(L, H), torch.nn.Linear(H, S)


def decode64(p64, z):
    h3 = torch.clamp_min(z @ p64["fc3.weight"].T + p64["fc3.bias"], 0)
    return torch.tanh(h3 @ p64["fc4.weight"].T + p64["fc4.bias"])


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def make(dims, precision, dev, seed=0):
    from rawaudiovae_kelsey_b200.model import VAE
    p64 = {k: v.double() for k, v in O.init_params(*dims, seed=seed).items()}
    torch.manual_seed(seed)
    m = VAE(*dims, precision=precision)
    m.load_state_dict({k: v.float() for k, v in p64.items()})
    return m.to(dev), p64


def padding_mask(flat):
    """True on every element of the flat buffers that belongs to no parameter."""
    pad = torch.ones(flat.total, dtype=torch.bool)
    for off, shape, strides in flat.geometry.values():
        rows, cols = (shape[0], shape[1]) if len(shape) == 2 else (1, shape[0])
        pitch = strides[0] if len(shape) == 2 else cols
        pad[off:off + rows * pitch].view(rows, pitch)[:, :cols] = False
    return pad.to(flat.params.device)


def assert_padding_zero(flat):
    pad = padding_mask(flat)
    assert int(pad.sum()) > 0
    bufs = {"params": flat.params, "grads": flat.grads, "exp_avg": flat.exp_avg, "exp_avg_sq": flat.exp_avg_sq,
            "shadow_hi": flat.shadow_hi.float()}
    if flat.shadow_lo is not None:
        bufs["shadow_lo"] = flat.shadow_lo.float()
    for k, b in bufs.items():
        assert int(torch.count_nonzero(b[pad])) == 0, k


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_forward_backward_parity(shape, precision, dev):
    from rawaudiovae_kelsey_b200.model import loss_function
    (S, H, L), _, B = shape
    tol = TOL[precision]
    model, p64 = make((S, H, L), precision, dev)
    g = torch.Generator().manual_seed(1)
    x = (torch.rand(B, S, generator=g) * 2 - 1) * 0.5
    eps = torch.randn(B, L, generator=g)
    xhat, mu, lv = model(x.to(dev), eps=eps.to(dev))
    assert xhat.shape == (B, S) and mu.shape == (B, L) and lv.shape == (B, L)
    loss = loss_function(xhat, x.to(dev), mu, lv, 0.5, S)
    loss.backward()
    act = O.forward(p64, x.double(), eps.double())
    assert rel(xhat, act["x_hat"]) < tol and rel(mu, act["mu"]) < tol and rel(lv, act["logvar"]) < tol
    ref_loss = O.loss_function(act["x_hat"], act["x"], act["mu"], act["logvar"], 0.5, S)
    assert abs(float(loss) - float(ref_loss)) <= tol * abs(float(ref_loss))
    # backward at the implementation's ReLU gates (test_gpu_parity.gated_reference), on the true columns
    plan = model._plan_for(B)
    m1 = (plan.activation("h1")[0][:, :H].float() > 0).cpu()
    m3 = (plan.activation("h3")[0][:, :H].float() > 0).cpu()
    for a, m in ((act["a1"], m1), (act["a3"], m3)):
        differ = m != (a > 0)
        assert bool((a.abs()[differ] <= tol * float(a.pow(2).mean().sqrt())).all())
    gref = O.backward(p64, act, 0.5, masks=(m1, m3))
    for k, p in model.named_parameters():
        assert p.grad.shape == p.shape
        assert rel(p.grad, gref[k]) < tol, k
    flat = model._flat
    pad = padding_mask(flat)
    assert int(torch.count_nonzero(flat.grads[pad])) == 0
    assert int(torch.count_nonzero(flat.params[pad])) == 0


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_three_adam_steps(shape, precision, dev):
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    (S, H, L), _, B = shape
    tol = TOL[precision]
    model, p64 = make((S, H, L), precision, dev)
    opt = Adam(model.parameters(), lr=1e-4)
    step = FusedTrainStep(model, opt, kl_beta=0.5, keep_grads=True)
    state = O.adam_init(p64)
    g = torch.Generator().manual_seed(2)
    for _ in range(3):
        x = (torch.rand(B, S, generator=g) * 2 - 1) * 0.5
        eps = torch.randn(B, L, generator=g)
        loss = float(step(x.to(dev), eps=eps.to(dev)))
        ref = O.train_step(p64, state, x.double(), eps.double(), 0.5, 1e-4)
        assert abs(loss - ref) <= tol * abs(ref)
    sd = model.state_dict()
    osd = opt.state_dict()["state"]
    for i, (k, p) in enumerate(model.named_parameters()):
        assert tuple(sd[k].shape) == tuple(p64[k].shape)
        assert rel(sd[k], p64[k]) < (1e-3 if precision == "fp32" else 1e-2), k
        assert rel(osd[i]["exp_avg"], state[k]["exp_avg"]) < 10 * tol, k
        assert rel(osd[i]["exp_avg_sq"], state[k]["exp_avg_sq"]) < 10 * tol, k
    torch.cuda.synchronize()
    assert_padding_zero(model._flat)
    # a checkpoint loads into a model of the true dims
    RefVAE(S, H, L).load_state_dict({k: v.cpu() for k, v in sd.items()})


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_philox_noise_matches_unpadded_draw(shape, dev):
    from rawaudiovae_kelsey_b200 import ops
    (S, H, L), _, B = shape
    model, _ = make((S, H, L), "bf16", dev)
    plan = model._plan_for(B)
    plan.load_batch(torch.zeros(B, S, device=dev))
    plan.gen_eps(1234, 7)
    torch.cuda.synchronize()
    full = ops.randn((B, L), 1234, 7, device=dev)
    assert torch.equal(plan.latent("eps"), full)
    # a data-parallel shard starting at row r0 = 3: its first element r0 * L is odd for L = 3 (inside a Philox block
    # of four), 48 for L = 16
    r0 = 3
    plan.load_batch(torch.zeros(B - r0, S, device=dev))
    plan.set_noise_rows(r0)
    plan.gen_eps(1234, 7)
    torch.cuda.synchronize()
    assert torch.equal(plan.latent("eps"), full[r0:])
    plan.set_noise_rows(0)
    # the same through rvae_randn: any element base, e.g. a batch of reconstruct_audio that starts at frame 50
    for base_row in (1, 50):
        part = ops.randn((B - base_row, L), 1234, 7, device=dev, elem_base=base_row * L)
        assert torch.equal(part, full[base_row:])


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_framing_gather_and_in_place(shape, dev):
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import FrameBatch
    (S, H, L), hop, B = shape
    rng = np.random.default_rng(3)
    audio = O.synth_wav(rng, hop * (B + 20)).astype(np.float32)
    ref = O.audio_dataset_frames(O.pad_to_multiple(audio, hop), S, hop)[:B]
    a = torch.from_numpy(audio).to(dev)
    f32, hi, _ = ops.frame_gather(a, B, hop, S, out_bf16=True)
    assert torch.equal(f32.cpu(), torch.from_numpy(np.ascontiguousarray(ref)).float())
    assert torch.equal(hi.cpu(), torch.from_numpy(np.ascontiguousarray(ref)).to(torch.bfloat16))
    # a run read in place (S % 8 == 0: bf16 mode) or gathered gives the same model outputs, bit for bit
    model, _ = make((S, H, L), "bf16", dev)
    eps = torch.randn(B, L, device=dev)
    fb = FrameBatch(a, B, hop, S)
    assert model._in_place(fb) == (S % 8 == 0)
    with torch.no_grad():
        out_run = model(fb, eps=eps)
        out_rows = model(f32, eps=eps)
    for u, v in zip(out_run, out_rows):
        assert torch.equal(u, v)


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_graph_prefetch_equals_eager(shape, dev):
    from rawaudiovae_kelsey_b200.model import FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    (S, H, L), hop, B = shape
    rng = np.random.default_rng(4)
    audio = torch.from_numpy(O.synth_wav(rng, hop * (8 * B + 20)).astype(np.float32)).to(dev)
    batches = [FrameBatch(audio, B, hop, S, first_frame=i * B) for i in range(6)]
    results = []
    for graph, pipelined in ((False, False), (True, True)):
        model, _ = make((S, H, L), "bf16", dev)
        model.eps_seed = 99
        opt = Adam(model.parameters(), lr=1e-4)
        step = FusedTrainStep(model, opt, kl_beta=0.5, graph=graph)
        losses = []
        for i, b in enumerate(batches):
            nxt = batches[i + 1] if pipelined and i + 1 < len(batches) else None
            losses.append(step(b, next_data=nxt).clone())
        torch.cuda.synchronize()
        if graph:
            assert step.stats["replays"] > 0
        results.append((torch.stack(losses), model._flat.params.clone()))
        assert_padding_zero(model._flat)
    # split-K weight gradients reduce-add in no fixed order: the tolerances of test_gpu_parity's graph / prefetch tests
    assert torch.allclose(results[0][0], results[1][0], rtol=1e-4, atol=0)
    assert rel(results[0][1], results[1][1]) < 1e-3


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_histograms_of_true_parameters(shape, dev):
    from rawaudiovae_kelsey_b200.stats import ParamHistogramLogger, default_bins

    class Sink:
        def __init__(self):
            self.rec = {}

        def add_histogram_raw(self, name, **kw):
            self.rec[name] = kw

    (S, H, L), _, _ = shape
    model, _ = make((S, H, L), "bf16", dev)
    sink = Sink()
    log = ParamHistogramLogger(model, sink)
    log.record(0)
    log.flush(wait=True)
    edges = np.asarray(default_bins(), dtype=np.float64)
    for name, p in model.named_parameters():
        v = p.detach().double().cpu().numpy().ravel()
        check_histogram(sink.rec[name], v, edges, name)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[0])))
def test_inference_api(shape, precision, dev):
    """encode_audio, decode_latents, lerp_latents, interpolate and reconstruct_audio (OLA and concat, and TestDataset
    framing) against the oracle, with batches that split the audio (batch_size 50: a batch's first Philox element
    lo * L is not a multiple of 4 for L = 3)."""
    from rawaudiovae_kelsey_b200 import inference as I
    from rawaudiovae_kelsey_b200 import ops
    (S, H, L), hop, _ = shape
    tol = TOL[precision]
    model, p64 = make((S, H, L), precision, dev)
    rng = np.random.default_rng(6)
    wav = O.synth_wav(rng, hop * 137 + 61).astype(np.float32)     # not a multiple of hop: zero-padded tail
    frames = torch.from_numpy(O.audio_dataset_frames(wav, S, hop)).double()
    N = frames.shape[0]
    mu, lv = I.encode_audio(model, wav, hop=hop, batch_size=50)
    act = O.forward(p64, frames, torch.zeros(N, L, dtype=torch.float64))
    assert mu.shape == lv.shape == (N, L)
    assert rel(mu, act["mu"]) < tol and rel(lv, act["logvar"]) < tol
    g = torch.Generator().manual_seed(7)
    z = torch.randn(N, L, generator=g)
    xd = I.decode_latents(model, z.to(dev), batch_size=50)
    assert xd.shape == (N, S) and rel(xd, decode64(p64, z.double())) < tol
    # interpolation between the encoding and its reverse, one alpha per frame (float64, as interp1d gives it)
    alpha = torch.linspace(0, 1, N, dtype=torch.float64)
    eps = torch.randn(N, L, generator=g)
    mb, lb = mu.flip(0).contiguous(), lv.flip(0).contiguous()
    a = alpha[:, None]
    m_ref = (1 - a) * mu.double().cpu() + a * mb.double().cpu()
    l_ref = (1 - a) * lv.double().cpu() + a * lb.double().cpu()
    z_ref = m_ref + eps.double() * torch.exp(0.5 * l_ref)
    zl, ml, ll = I.lerp_latents(mu, lv, mb, lb, alpha.to(dev), eps.to(dev), return_dist=True)
    assert zl.shape == (N, L)
    assert rel(ml, m_ref) < 1e-6 and rel(ll, l_ref) < 1e-6 and rel(zl, z_ref) < 1e-5
    xi = I.interpolate(model, mu, lv, mb, lb, alpha.to(dev), eps=eps.to(dev), batch_size=50)
    assert xi.shape == (N, S) and rel(xi, decode64(p64, z_ref)) < tol
    # reconstruction with the library's Philox noise: the batches draw pieces of ONE [N, L] noise tensor
    for mode in ("ola", "concat"):
        model.eps_seed, model._eps_counter = 11, 0
        out = I.reconstruct_audio(model, wav, hop=hop, mode=mode, batch_size=50)
        e = ops.randn((N, L), 11, 0, device=dev).double().cpu()
        xh = O.forward(p64, frames, e)["x_hat"].numpy()
        ref = O.resynth_overlap_add(xh, hop) if mode == "ola" else O.resynth_concat(xh)
        assert tuple(out.shape) == ref.shape, mode
        assert rel(out, torch.from_numpy(ref)) < tol, mode
    model.eps_seed, model._eps_counter = 11, 0
    out = I.reconstruct_audio(model, wav, batch_size=50)          # TestDataset framing, concatenated
    tframes = torch.from_numpy(O.test_dataset_frames(wav, S)).double()
    e = ops.randn((tframes.shape[0], L), 11, 0, device=dev).double().cpu()
    ref = O.resynth_concat(O.forward(p64, tframes, e)["x_hat"].numpy())
    assert tuple(out.shape) == ref.shape and rel(out, torch.from_numpy(ref)) < tol


def test_fp32_frames_gathered_into_padded_rows(dev):
    """fp32 mode with a padded segment_length gathers frames (its residual plane of x is read from memory, so the
    zeros past S must be real): steps on FrameBatch input against the oracle loop, then a prefetching run."""
    from rawaudiovae_kelsey_b200.model import FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    (S, H, L), hop, B = SHAPES[0]
    model, p64 = make((S, H, L), "fp32", dev)
    step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-4), kl_beta=0.5, keep_grads=True)
    state = O.adam_init(p64)
    rng = np.random.default_rng(8)
    wav = O.synth_wav(rng, hop * (8 * B + 20)).astype(np.float32)
    audio = torch.from_numpy(wav).to(dev)
    frames = torch.from_numpy(O.audio_dataset_frames(wav, S, hop)).double()
    g = torch.Generator().manual_seed(9)
    for i in range(2):
        fb = FrameBatch(audio, B, hop, S, first_frame=i * B)
        assert fb.span and not model._in_place(fb)
        eps = torch.randn(B, L, generator=g)
        loss = float(step(fb, eps=eps.to(dev)))
        ref = O.train_step(p64, state, frames[i * B:(i + 1) * B], eps.double(), 0.5, 1e-4)
        assert abs(loss - ref) <= 1e-4 * abs(ref)
    for k, p in model.state_dict().items():
        assert rel(p, p64[k]) < 1e-3, k
    torch.cuda.synchronize()
    assert_padding_zero(model._flat)
    # the next batch gathered by the background stream (prefetch), Philox noise: equal to plain steps
    batches = [FrameBatch(audio, B, hop, S, first_frame=i * B) for i in range(5)]
    results = []
    for pipelined in (False, True):
        m, _ = make((S, H, L), "fp32", dev)
        m.eps_seed = 5
        st = FusedTrainStep(m, Adam(m.parameters(), lr=1e-4), kl_beta=0.5)
        losses = [st(b, next_data=batches[i + 1] if pipelined and i + 1 < len(batches) else None).clone()
                  for i, b in enumerate(batches)]
        torch.cuda.synchronize()
        assert_padding_zero(m._flat)
        results.append((torch.stack(losses), m._flat.params.clone()))
    assert torch.allclose(results[0][0], results[1][0], rtol=1e-4, atol=0)
    assert rel(results[0][1], results[1][1]) < 1e-3


def _trainer_config(path, data, *, S, H, L, hop, batch, extra):
    from test_gpu_parity import _trainer_ini
    _trainer_ini(path, data, batch=batch, extra_training=extra)
    text = path.read_text()
    for a, b in (("hop_length = 128", f"hop_length = {hop}"), ("segment_length = 1024", f"segment_length = {S}"),
                 ("latent_dim = 64", f"latent_dim = {L}"), ("n_units = 256", f"n_units = {H}")):
        assert a in text
        text = text.replace(a, b)
    path.write_text(text)


def _check_trainer_run(data, dims):
    """The last ckpt_* loads into the reference module of the true dims, and the last histogram events equal
    make_histogram of that checkpoint's parameters (num = the true element count)."""
    from test_gpu_param_histograms import _events
    from rawaudiovae_kelsey_b200.stats import default_bins
    run = next((data / "unit-test").glob("run-*"))
    _, hist, _ = _events(run)
    last = sorted((run / "model" / "checkpoints").glob("ckpt_*"))[-1]
    sd = torch.load(last, map_location="cpu", weights_only=False)["state_dict"]
    RefVAE(*dims).load_state_dict(sd)
    h = hist[max(hist)]
    assert len(h) == 10
    edges = np.asarray(default_bins(), dtype=np.float64)
    for name, v in sd.items():
        pb = h[name]
        check_histogram({"bucket_limits": list(pb.bucket_limit), "bucket_counts": list(pb.bucket), "min": pb.min,
                         "max": pb.max, "num": pb.num, "sum": pb.sum, "sum_squares": pb.sum_squares},
                        v.numpy(), edges, name)
        assert pb.num == v.numel(), name


def test_epoch_trainer_at_padded_dims(dev, tmp_path):
    """train.py with n_units = 300, latent_dim = 16, segment_length = 1000, hop_length = 200."""
    from test_gpu_param_histograms import _corpus
    from rawaudiovae_kelsey_b200 import trainer
    data = _corpus(tmp_path)
    ini = tmp_path / "e.ini"
    _trainer_config(ini, data, S=1000, H=300, L=16, hop=200, batch=200,
                    extra="epochs = 2\nsave_best_model_after = 1\ncheckpoint_interval = 1")
    assert trainer.run_epoch_trainer(["--config", str(ini)]) in (0, None)
    _check_trainer_run(data, (1000, 300, 16))


def test_stream_trainer_at_padded_dims(dev, tmp_path):
    """train_iterable.py with n_units = 2000, latent_dim = 16 (segment_length stays 1024, as the reference's stream
    frames at 1024 samples)."""
    from test_gpu_param_histograms import _corpus
    from rawaudiovae_kelsey_b200 import trainer
    data = _corpus(tmp_path)
    ini = tmp_path / "s.ini"
    _trainer_config(ini, data, S=1024, H=2000, L=16, hop=128, batch=200,
                    extra="epochs = 1\ntotal_num_frames = 2000\ncheckpoint_interval = 4\nlog_interval = 3\n"
                          "histogram_interval = 1")
    assert trainer.run_stream_trainer(["--config", str(ini)]) in (0, None)
    _check_trainer_run(data, (1024, 2000, 16))
