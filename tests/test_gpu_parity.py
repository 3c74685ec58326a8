"""GPU parity tests (-m gpu): the sm_100a path, called through the C ABI, against the CPU oracle and the committed
golden vectors of the reference. Tolerances are BASELINE.json's: frame indices bit-exact; fp32 mode <= 1e-4
relative; bf16 mode <= 2e-2 relative; loss curves within 1 % over 1k steps."""
import json

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

BF16_TOL = 2e-2        # bf16 mode vs the reference (BASELINE.json)
FP32_TOL = 1e-4        # fp32 mode vs the reference (BASELINE.json)
BF16_EMU_TOL = 5e-3    # bf16 mode vs the oracle run with bf16-rounded GEMM operands (same rounding points)


def rel(a, b):
    a = torch.as_tensor(a).detach().double().cpu().flatten()
    b = torch.as_tensor(b).detach().double().cpu().flatten()
    return float((a - b).norm() / (b.norm() + 1e-300))


def gated_reference(model, p64, x, eps, beta, tol):
    """The reference's arithmetic in fp64 (oracle), with its backward evaluated at the IMPLEMENTATION's ReLU gates.

    A ReLU gate [a > 0] is ill-conditioned at a ~ 0: any rounding of the pre-activation flips it, and a flipped gate
    changes that unit's gradient by 100 %, so a plain tensor-norm comparison of gradients measures how many
    near-zero units exist, not kernel accuracy (fp32 cuBLAS vs fp64 shows the same effect). The check is therefore
    split in two, both at the mode's tolerance `tol`:
      (1) the implementation's gates differ from the reference's only on units whose reference pre-activation lies
          within tol * rms(a) of zero (i.e. the pre-activations are accurate to tol), and
      (2) given identical gates, every gradient is within tol (relative L2) of the reference.
    Must be called right after the implementation's backward (reads h1 / h3 from the plan workspace)."""
    from oracle import rawvae_oracle as O
    act = O.forward(p64, x.double().cpu(), eps.double().cpu())
    plan = model._plan_for(act["x"].shape[0])
    assert plan.batch == act["x"].shape[0]
    m1 = (plan.activation("h1")[0].float() > 0).cpu()
    m3 = (plan.activation("h3")[0].float() > 0).cpu()
    flips = 0
    for a, m, name in ((act["a1"], m1, "h1"), (act["a3"], m3, "h3")):
        differ = m != (a > 0)
        band = tol * float(a.pow(2).mean().sqrt())
        assert bool((a.abs()[differ] <= band).all()), f"{name}: a gate differs outside the +-{band:.2e} band"
        flips += int(differ.sum())
    return act, O.backward(p64, act, beta, masks=(m1, m3)), flips


def bf16_oracle_grads(params64, x, eps, beta):
    from oracle import rawvae_oracle as O
    act = O.forward(params64, x.double(), eps.double(), O.bf16_operands)
    return O.backward(params64, act, beta, 1.0, O.bf16_operands), act


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from rawaudiovae_kelsey_b200 import _lib
    assert _lib.library_path().exists(), "librvae_b200.so missing - the CUDA extension must be built in-tree"
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def small(golden_dir):
    from oracle import gen_golden
    return gen_golden.load_small(golden_dir)


def make_model(small, prefix, dev, precision):
    from rawvae.model import VAE
    from oracle.rawvae_oracle import PARAM_NAMES
    S, H, L, B, steps = (int(v) for v in small["meta"])
    m = VAE(S, H, L, precision=precision)
    m.load_state_dict({k: torch.from_numpy(small[f"{prefix}/{k}"]) for k in PARAM_NAMES})
    return m.to(dev)


# ------------------------------------------------------------------------------------------------ golden, small dims
@pytest.mark.parametrize("precision,tol", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_forward_backward_vs_reference_golden(dev, small, precision, tol):
    from rawvae.model import loss_function
    from oracle.rawvae_oracle import PARAM_NAMES
    S, H, L, B, steps = (int(v) for v in small["meta"])
    kl_beta, lr = (float(v) for v in small["hyper"])
    model = make_model(small, "init", dev, precision)
    x = torch.from_numpy(small["x"]).to(dev)
    eps = torch.from_numpy(small["eps"][0]).to(dev)
    xh, mu, lv = model(x, eps=eps)
    assert xh.shape == (B, S) and mu.shape == (B, L) and lv.shape == (B, L)
    assert rel(xh, small["x_hat"]) < tol
    assert rel(mu, small["mu"]) < tol
    assert rel(lv, small["logvar"]) < tol
    loss = loss_function(xh, x, mu, lv, kl_beta, S)
    assert loss.dim() == 0
    assert abs(loss.item() - float(small["losses"][0])) < tol * abs(float(small["losses"][0]))
    loss.backward()
    assert all(p.grad is not None for p in model.parameters())
    p64 = {k: torch.from_numpy(small["init/" + k]).double() for k in PARAM_NAMES}
    xs, es = torch.from_numpy(small["x"]), torch.from_numpy(small["eps"][0])
    act, gref, flips = gated_reference(model, p64, xs, es, kl_beta, tol)
    for k, p in model.named_parameters():
        assert rel(p.grad, gref[k]) < tol, k
        if flips == 0:                       # identical gating: compare with the reference's own gradients directly
            assert rel(p.grad, small["grad/" + k]) < tol, k
    if precision == "bf16":
        emu, _ = bf16_oracle_grads(p64, xs, es, kl_beta)
        for k, p in model.named_parameters():
            assert rel(p.grad, emu[k]) < BF16_EMU_TOL, k


@pytest.mark.parametrize("precision,tol", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_three_adam_steps_vs_reference_golden(dev, small, precision, tol):
    """The reference loop body (train_iterable.py:200-210) through the drop-in API, 3 steps: per-step losses against
    the reference's golden losses; Adam moments after the FIRST step against the gated reference gradient (m = 0.1 g,
    v = 0.001 g^2 exactly); optimizer state layout and final weights against the reference's."""
    from rawvae.model import loss_function
    from rawaudiovae_kelsey_b200.optim import Adam
    from oracle import rawvae_oracle as O
    S, H, L, B, steps = (int(v) for v in small["meta"])
    kl_beta, lr = (float(v) for v in small["hyper"])
    model = make_model(small, "init", dev, precision)
    opt = Adam(model.parameters(), lr=lr)
    x = torch.from_numpy(small["x"]).to(dev)
    p64 = {k: torch.from_numpy(small["init/" + k]).double() for k in O.PARAM_NAMES}
    for s in range(steps):
        opt.zero_grad()
        xh, mu, lv = model(x, eps=torch.from_numpy(small["eps"][s]).to(dev))
        loss = loss_function(xh, x, mu, lv, kl_beta, S)
        loss.backward()
        if s == 0:
            _, gref, _ = gated_reference(model, p64, torch.from_numpy(small["x"]), torch.from_numpy(small["eps"][0]),
                                         kl_beta, tol)
        opt.step()
        assert abs(loss.item() - float(small["losses"][s])) < tol * abs(float(small["losses"][s]))
        if s == 0:
            st0 = opt.state_dict()["state"]
            for i, (k, _) in enumerate(model.named_parameters()):
                assert rel(st0[i]["exp_avg"], 0.1 * gref[k]) < tol, k
                assert rel(st0[i]["exp_avg_sq"], 0.001 * gref[k] ** 2) < 2 * tol, k
    ost = opt.state_dict()
    assert sorted(ost["state"][0].keys()) == ["exp_avg", "exp_avg_sq", "step"]
    assert float(ost["state"][0]["step"]) == steps
    assert len(ost["state"]) == 10 and ost["param_groups"][0]["params"] == list(range(10))
    sd = model.state_dict()
    for i, k in enumerate(sd):
        # weights moved by ~3 lr (~6 % of their norm); Adam's m/sqrt(v) ~ sign(g) amplifies rounding of near-zero
        # gradient entries, so the bound is on the weights, not on the update
        assert rel(sd[k], small["final/" + k]) < (1e-3 if precision == "fp32" else 1e-2), k
        # after 3 steps trajectories have separated by rounding noise (gates, bf16 weight shadows): loose bound
        assert rel(ost["state"][i]["exp_avg"], small["exp_avg/" + k]) < (1e-2 if precision == "fp32" else 8e-2), k


@pytest.mark.parametrize("precision,tol", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_fused_train_step_matches_oracle(dev, small, precision, tol):
    """rvae_plan_train_step (one C call per step: fused loss epilogues, backward, Adam): loss per step against the
    reference's golden losses; first-step Adam moments against the gated reference gradient."""
    from rawvae.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from oracle import rawvae_oracle as O
    S, H, L, B, steps = (int(v) for v in small["meta"])
    kl_beta, lr = (float(v) for v in small["hyper"])
    model = make_model(small, "init", dev, precision)
    opt = Adam(model.parameters(), lr=lr)
    step = FusedTrainStep(model, opt, kl_beta, keep_grads=(precision == "fp32"))  # both gradient-buffer policies
    p64 = {k: torch.from_numpy(small["init/" + k]).double() for k in O.PARAM_NAMES}
    x = torch.from_numpy(small["x"])
    flat = model._flat
    for s in range(steps):
        eps = torch.from_numpy(small["eps"][s])
        loss = step(x.to(dev), eps=eps.to(dev))
        assert abs(loss.item() - float(small["losses"][s])) < tol * float(small["losses"][s])
        if s == 0:
            _, gref, _ = gated_reference(model, p64, x, eps, kl_beta, tol)
            for k in O.PARAM_NAMES:
                if step.keep_grads:
                    assert rel(flat.view(flat.grads, k), gref[k]) < tol, k
                else:
                    assert float(flat.view(flat.grads, k).abs().max()) == 0.0, k   # cleared by the Adam kernel
                assert rel(flat.view(flat.exp_avg, k), 0.1 * gref[k]) < tol, k
    assert float(flat.step) == steps
    # bf16 shadow planes follow the fp32 master weights
    assert rel(flat.shadow_hi.float(), flat.params) < 4e-3
    for k in O.PARAM_NAMES:
        assert rel(flat.view(flat.params, k), small["final/" + k]) < (1e-3 if precision == "fp32" else 1e-2), k


def test_default_ini_dims_fused_step(dev, golden_dir):
    """default.ini dimensions (S=1024, H=2048, L=256), B=256: loss and gradient norms against the reference's
    summary; weights regenerated from the seed exactly as the reference does (torch.manual_seed(0); VAE(...))."""
    from rawvae.model import VAE, loss_function
    g = json.loads((golden_dir / "model_default_summary.json").read_text())
    S, H, L, B = g["S"], g["H"], g["L"], g["B"]
    torch.manual_seed(0)
    model = VAE(S, H, L).to(dev)
    assert sum(p.numel() for p in model.parameters()) == g["n_params"]
    assert list(model.state_dict().keys()) == g["state_dict_keys"]
    gen = torch.Generator().manual_seed(1)
    x = (torch.rand(B, S, generator=gen) * 2 - 1).to(dev)
    eps = torch.randn(B, L, generator=gen).to(dev)
    for precision, tol in (("bf16", BF16_TOL), ("fp32", FP32_TOL)):
        model.set_precision(precision)
        model.zero_grad()
        xh, mu, lv = model(x, eps=eps)
        loss = loss_function(xh, x, mu, lv, g["kl_beta"], S)
        loss.backward()
        assert abs(loss.item() - g["losses"][0]) < tol * g["losses"][0]
        for name, t in (("x_hat", xh), ("mu", mu), ("logvar", lv)):
            assert abs(float(t.double().norm()) - g[name]["norm"]) < tol * g[name]["norm"], name
        for k, p in model.named_parameters():
            assert abs(float(p.grad.double().norm()) - g["grads"][k]["norm"]) < tol * g["grads"][k]["norm"], k


# ------------------------------------------------------------------------------------------------ larger, oracle on the fly
@pytest.mark.parametrize("precision,tol", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_activations_and_gradients_vs_oracle_ragged_batch(dev, precision, tol):
    """A ragged batch (B=300, not a multiple of the 128-row tile) at S=256, H=320, L=64: every activation and
    gradient tensor against the fp64 oracle."""
    from rawvae.model import VAE, loss_function
    from oracle import rawvae_oracle as O
    S, H, L, B, beta = 256, 320, 64, 300, 1e-2
    torch.manual_seed(3)
    model = VAE(S, H, L, precision=precision).to(dev)
    p64 = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    gen = torch.Generator().manual_seed(5)
    x = torch.rand(B, S, generator=gen) * 2 - 1
    eps = torch.randn(B, L, generator=gen)
    xh, mu, lv = model(x.to(dev), eps=eps.to(dev))
    loss = loss_function(xh, x.to(dev), mu, lv, beta, S)
    loss.backward()
    act, gref, flips = gated_reference(model, p64, x, eps, beta, tol)
    ref_loss = O.loss_function(act["x_hat"], act["x"], act["mu"], act["logvar"], beta, S)
    assert rel(xh, act["x_hat"]) < tol and rel(mu, act["mu"]) < tol and rel(lv, act["logvar"]) < tol
    assert abs(loss.item() - float(ref_loss)) < tol * float(ref_loss)
    for k, prm in model.named_parameters():
        assert rel(prm.grad, gref[k]) < tol, k
    if precision == "bf16":
        emu, emu_act = bf16_oracle_grads(p64, x, eps, beta)
        assert rel(xh, emu_act["x_hat"]) < BF16_EMU_TOL and rel(mu, emu_act["mu"]) < BF16_EMU_TOL
        for k, prm in model.named_parameters():
            assert rel(prm.grad, emu[k]) < BF16_EMU_TOL, k


def test_loss_curve_1k_steps_within_one_percent(dev):
    """1000 optimizer steps of the default.ini VAE (S=1024, H=2048, L=256; lr and kl_beta as shipped) on synthetic
    sine+noise frames, a fresh batch and fresh eps every step: the bf16 fused path's loss curve stays within 1 % of
    the reference algorithm run in fp32 on the CPU (the oracle port), step by step (BASELINE.json north_star)."""
    from rawvae.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from oracle import rawvae_oracle as O
    S, H, L, B, n = 1024, 2048, 256, 128, 1000
    kl_beta, lr, hop = 1e-4, 1e-4, 128
    rng = np.random.default_rng(1234)
    audio = np.concatenate([O.synth_wav(rng, 44100 * 2) for _ in range(4)])
    frames = torch.from_numpy(O.audio_dataset_frames(audio, S, hop))
    gen = torch.Generator().manual_seed(11)
    idx = torch.randint(0, len(frames), (n, B), generator=gen)
    eps_all = torch.randn(n, B, L, generator=gen)
    torch.manual_seed(0)
    model = VAE(S, H, L).to(dev)
    p = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}       # fp32, as the reference trains
    st = O.adam_init(p)
    opt = Adam(model.parameters(), lr=lr)
    step = FusedTrainStep(model, opt, kl_beta, ring=n)
    frames_dev, eps_dev, idx_dev = frames.to(dev), eps_all.to(dev), idx.to(dev)
    torch.set_num_threads(max(1, torch.get_num_threads()))
    ref = []
    for s in range(n):
        step(frames_dev[idx_dev[s]], eps=eps_dev[s])
        ref.append(O.train_step(p, st, frames[idx[s]], eps_all[s], kl_beta, lr))
    got = step.ring.cpu().double().numpy()
    ref = np.array(ref)
    err = np.abs(got - ref) / ref
    assert ref[-50:].mean() < 0.9 * ref[:50].mean(), "the reference should be learning"
    assert err.max() < 0.01, f"max loss-curve deviation {err.max():.4f} at step {err.argmax()}"


# ------------------------------------------------------------------------------------------------ framing / resynthesis
def test_framing_bit_exact_vs_reference_golden(dev, golden_dir):
    from rawaudiovae_kelsey_b200 import ops
    from rawvae.dataset import AudioDataset, TestDataset
    ds = np.load(golden_dir / "dataset.npz")
    for n in (22087, 1024, 1025, 2048, 1151, 1152):
        audio = ds[f"audio_{n}"]
        a = AudioDataset(audio, 1024, 44100, 128)
        t = TestDataset(audio, 1024, 44100)
        assert [len(a), len(t)] == [int(v) for v in ds[f"audio_len_{n}"]]
        idx = torch.from_numpy(ds[f"audio_idx_{n}"]).to(dev)
        ad = torch.from_numpy(audio).to(dev)                       # un-padded: the kernel zero-fills the tail
        f32, hi, _ = ops.frame_gather(ad, len(idx), 128, 1024, frame_idx=idx, out_bf16=True)
        np.testing.assert_array_equal(f32.cpu().numpy(), ds[f"audio_frames_{n}"])
        assert torch.equal(hi.cpu(), torch.from_numpy(ds[f"audio_frames_{n}"]).to(torch.bfloat16))
        tf, _, _ = ops.frame_gather(ad, len(t), 1024, 1024)
        np.testing.assert_array_equal(tf.cpu().numpy(), ds[f"test_frames_{n}"])


def test_gpu_stream_matches_reference_stream(dev, golden_dir, tmp_path):
    """GpuFrameStream over the same three wavs reproduces the reference IterableAudioDataset stream bit-exactly
    (stereo -> channel 0, zero padding, batches straddling files, endless cycling)."""
    import scipy.io.wavfile as wavfile
    from rawvae.dataset import IterableAudioDataset
    from rawaudiovae_kelsey_b200 import ops
    ds = np.load(golden_dir / "dataset.npz")
    order = [str(s) for s in ds["stream_order"]]
    for name in order:
        wavfile.write(str(tmp_path / name), 44100, ds["stream_pcm_" + name])
    it = IterableAudioDataset(tmp_path, 44100, 128, torch.float32, dev, shuffle=False)
    it.audio_file_list = [tmp_path / n for n in order]             # glob order is filesystem dependent
    got = []
    for fb in it.gpu_stream(batch_size=50):
        got.append(fb.materialize())
        if sum(len(g) for g in got) >= 150:
            break
    got = torch.cat(got)[:150].cpu().numpy()
    np.testing.assert_array_equal(got, ds["stream_frames"])
    # PCM16 on the wire / in the ring decodes to the same floats
    got16 = []
    stream16 = it.gpu_stream(batch_size=50, pcm16=True)
    for fb in stream16:
        got16.append(fb.materialize())
        if sum(len(g) for g in got16) >= 150:
            break
    np.testing.assert_array_equal(torch.cat(got16)[:150].cpu().numpy(), ds["stream_frames"])
    assert stream16.ring.dtype == torch.int16


def _write_mixed_corpus(root):
    """14 short wavs: 44.1 kHz mono, 48 kHz and 22.05 kHz (resampled on ingest), one stereo (channel 0 is kept)."""
    import scipy.io.wavfile as wavfile
    from oracle.rawvae_oracle import synth_wav
    rng = np.random.default_rng(11)
    names = []
    for i in range(14):
        rate = (44100, 48000, 44100, 22050, 44100, 44100, 44100)[i % 7]
        secs = 0.3 + 0.2 * rng.random()
        x = np.round(synth_wav(rng, int(rate * secs), rate) * 32767).astype(np.int16)
        if i == 4:
            x = np.stack([x, x[::-1]], axis=1)
        wavfile.write(str(root / f"f{i:02d}.wav"), rate, x)
        names.append(root / f"f{i:02d}.wav")
    return names


def test_gpu_stream_ring_smaller_than_corpus_and_resampled_file(dev, tmp_path):
    """SURVEY.md 8f N2: a corpus LARGER than the ingest ring streams through it (regions are overwritten only after
    their readers ran, files still resident are not uploaded again), a 48 kHz file is resampled to the training rate
    exactly as the reference does (rawvae/dataset.py:50-51: torchaudio.functional.resample), a stereo file keeps
    channel 0 - and every frame equals the CPU IterableAudioDataset stream's frame, bit for bit, over several cycles."""
    import scipy.io.wavfile as wavfile
    from itertools import islice
    from rawvae.dataset import IterableAudioDataset
    from oracle.rawvae_oracle import synth_wav
    names = _write_mixed_corpus(tmp_path)
    sr = 44100
    ds = IterableAudioDataset(tmp_path, sr, 128, torch.float32, "cpu", shuffle=False)
    ds.audio_file_list = names
    B, n_batches = 32, 200                                 # ~3 cycles over the files
    want = torch.stack(list(islice(iter(ds), B * n_batches))).numpy()
    total = sum(ds.load_file(f).numel() for f in names)
    stream = ds.gpu_stream(batch_size=B, device=dev)
    stream.capacity = int(0.4 * total) // 1024 * 1024      # the ring holds less than half of the corpus
    got = torch.cat([fb.materialize() for fb in islice(iter(stream), n_batches)]).cpu().numpy()
    np.testing.assert_array_equal(got, want)
    assert stream.stats["ring_wraps"] >= 3 and stream.stats["files_uploaded"] > len(names)
    assert stream.ring.numel() * 4 < total * 4
    # a ring that holds everything uploads each file once and then serves it from HBM
    big = ds.gpu_stream(batch_size=B, device=dev)
    got2 = torch.cat([fb.materialize() for fb in islice(iter(big), n_batches)]).cpu().numpy()
    np.testing.assert_array_equal(got2, want)
    assert big.stats["files_uploaded"] == len(names) and big.stats["resident_hits"] > len(names)


def test_full_size_framing_roundtrip_and_checksum(dev):
    """Config-sized property test: 60 s of 44.1 kHz audio -> 20 657 overlapping frames -> overlap-add == padded
    input; concat of TestDataset frames == padded input; checksum of frames == weighted checksum of samples."""
    from rawaudiovae_kelsey_b200 import ops
    from oracle.rawvae_oracle import audio_dataset_len
    n, S, hop = 44100 * 60 + 77, 1024, 128
    gen = torch.Generator().manual_seed(9)
    audio = (torch.rand(n, generator=gen) * 2 - 1).to(dev)
    N = audio_dataset_len(n, S, hop)
    frames, _, _ = ops.frame_gather(audio, N, hop, S)
    P = -(-n // hop) * hop
    pad = torch.cat([audio, torch.zeros(P - n, device=dev)])
    assert torch.equal(frames, pad.unfold(0, S, hop))
    ola = ops.overlap_add(frames, hop)
    assert ola.numel() == P and float((ola - pad).abs().max()) < 1e-6
    cnt = torch.ones(P, dtype=torch.float64, device=dev)
    cover = torch.minimum(torch.arange(P, device=dev) // hop, torch.tensor(N - 1, device=dev)) - \
        torch.clamp((torch.arange(P, device=dev) - S + hop) // hop, min=0) + 1
    assert abs(float(frames.double().sum()) - float((pad.double() * cover.double() * cnt).sum())) < 1e-6 * N
    PT = -(-n // S) * S
    tf, _, _ = ops.frame_gather(audio, PT // S, S, S)
    assert torch.equal(tf.view(-1), torch.cat([audio, torch.zeros(PT - n, device=dev)]))
    assert torch.equal(ops.overlap_add(tf, S), tf.view(-1))


def test_overlap_add_vector_scalar_and_ragged_paths(dev):
    """The float4 path (S, hop multiples of 4), its < 4-sample ragged tail, the scalar path (odd hop) and a
    truncated / over-long output length all follow the oracle's rule; vector and scalar paths agree bit for bit."""
    from rawaudiovae_kelsey_b200 import ops
    from oracle import rawvae_oracle as O
    gen = torch.Generator().manual_seed(11)
    for n_frames, S, hop in [(37, 64, 16), (37, 64, 12), (19, 60, 15), (5, 64, 64), (1, 32, 8), (23, 128, 6)]:
        fr = torch.randn(n_frames, S, generator=gen)
        ref = torch.from_numpy(O.resynth_overlap_add(fr.numpy(), hop)).float()
        full = (n_frames - 1) * hop + S
        for n_out in (full, full - 1, full - 3, full + 5, 3):
            got = ops.overlap_add(fr.to(dev), hop, n_out).cpu()
            want = torch.zeros(n_out)
            k = min(n_out, full)
            want[:k] = ref[:k]
            assert got.shape == want.shape and torch.allclose(got, want, atol=1e-6), (n_frames, S, hop, n_out)
        # a misaligned view forces the scalar path: same bits as the vector path
        if S % 4 == 0 and hop % 4 == 0:
            buf = torch.empty(n_frames * S + 1, device=dev)
            buf[1:] = fr.view(-1).to(dev)
            assert torch.equal(ops.overlap_add(buf[1:].view(n_frames, S), hop), ops.overlap_add(fr.to(dev), hop))


# ------------------------------------------------------------------------------------------------ full-size properties
def test_full_size_gradient_additivity_and_api_agreement(dev):
    """BASELINE config (default.ini dims, 8192 frames): size-independent properties instead of an 8192-row oracle run.
    (1) fused step gradients == autograd-API gradients (two different kernel routes to the same numbers);
    (2) with global-batch normalisation, grad(batch) == grad(first half) + grad(second half): the identity data
        parallelism relies on."""
    from rawvae.model import VAE, loss_function
    S, H, L, B, beta = 1024, 2048, 256, 8192, 1e-4
    torch.manual_seed(0)
    model = VAE(S, H, L).to(dev)
    gen = torch.Generator().manual_seed(2)
    x = (torch.rand(B, S, generator=gen) * 2 - 1).to(dev)
    eps = torch.randn(B, L, generator=gen).to(dev)
    xh, mu, lv = model(x, eps=eps)
    loss = loss_function(xh, x, mu, lv, beta, S)
    loss.backward()
    g_api = model._flat.grads.clone()
    api_loss = loss.item()

    plan = model._plan_for(B)

    def fused(xs, es, global_batch):
        plan.load_batch(xs)
        plan.set_eps(es)
        plan.set_global_batch(global_batch)
        plan.forward(beta, fused_loss=True, want_xhat=False)
        out = torch.zeros(1, device=dev)
        plan.finish_loss(beta, out)
        plan.backward(-1)
        plan.set_global_batch(0)
        return model._flat.grads.clone(), out.item()

    step0 = float(model._flat.step)
    g_full, l_full = fused(x, eps, 0)
    assert abs(l_full - api_loss) < 1e-3 * api_loss
    assert rel(g_full, g_api) < 5e-3          # same bf16 operands; the API route stages g_xhat in fp32 first
    g_a, l_a = fused(x[: B // 2], eps[: B // 2], B)
    g_b, l_b = fused(x[B // 2:], eps[B // 2:], B)
    assert abs(0.5 * (l_a + l_b) - l_full) < 1e-5 * l_full   # reported losses are per-shard means
    assert rel(g_a + g_b, g_full) < 1e-3
    model._flat.step.fill_(step0)             # finish_loss bumps the Adam step counter; restore
    assert 0.2 < api_loss < 0.6               # init-time loss on U(-1,1) input is ~0.3855 (SURVEY.md 8c)


def test_cuda_graph_step_equals_eager_step(dev):
    """FusedTrainStep(graph=True) replays a captured CUDA graph of the step; frame indices, Philox offset and
    loss-ring slot are read from device memory, so 12 replayed steps match 12 eagerly enqueued steps."""
    from rawvae.model import VAE, FusedTrainStep, FrameBatch
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, B, hop, n = 256, 320, 64, 384, 64, 12
    gen = torch.Generator().manual_seed(4)
    audio = (torch.rand(200000, generator=gen) * 2 - 1).to(dev)
    n_frames = (audio.numel() - S) // hop + 1
    idx = torch.randint(0, n_frames, (n, B), generator=gen).to(dev)
    losses = {}
    for use_graph in (False, True):
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        model.eps_seed = 77
        opt = Adam(model.parameters(), lr=1e-3)
        step = FusedTrainStep(model, opt, 1e-3, ring=16, graph=use_graph)
        out = []
        for i in range(n):
            fb = FrameBatch(audio, B, hop, S, frame_idx=idx[i]) if i % 3 else \
                FrameBatch(audio, B, hop, S, first_frame=int(idx[i, 0]))        # sequential batches use the same graph
            out.append(step(fb).clone())
        losses[use_graph] = torch.stack(out).cpu()
        if use_graph:
            # one graph per input layout: gathered index batches, and runs read in place (FrameBatch.span)
            assert len(step._graphs) == 2 and step.stats["captures"] == 2
        final = model._flat.params.clone()
        losses[("w", use_graph)] = final
    assert torch.allclose(losses[True], losses[False], rtol=1e-4, atol=0)
    # weights: the split-K reduce-adds and bias-gradient atomics land in a timing-dependent order, and Adam's
    # normalised update turns that fp32 reassociation noise in near-zero gradient entries into O(lr) differences
    assert rel(losses[("w", True)], losses[("w", False)]) < 1e-3
    assert float(losses[False][-1]) < float(losses[False][0])


@pytest.mark.parametrize("use_graph", [False, True])
def test_prefetched_steps_equal_plain_steps(dev, use_graph):
    """Pipelined input path: step(data, next_data=...) gathers the next batch and draws its noise on the background
    stream while the current step runs (double-buffered inputs); the losses and weights match the plain path, where
    every step loads its own batch - same frames, same Philox noise (offset = device step counter)."""
    from rawvae.model import VAE, FusedTrainStep, FrameBatch
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, B, hop, n = 256, 320, 64, 384, 64, 14
    gen = torch.Generator().manual_seed(5)
    audio = (torch.rand(150000, generator=gen) * 2 - 1).to(dev)
    n_frames = (audio.numel() - S) // hop + 1
    idx = torch.randint(0, n_frames, (n, B), generator=gen).to(dev)
    batches = [FrameBatch(audio, B, hop, S, frame_idx=idx[i]) if i % 4 else
               FrameBatch(audio, B, hop, S, first_frame=int(idx[i, 0]) % (n_frames - B)) for i in range(n)]
    res = {}
    for mode in ("plain", "pipelined"):
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        model.eps_seed = 99
        opt = Adam(model.parameters(), lr=1e-3)
        step = FusedTrainStep(model, opt, 1e-3, ring=16, graph=use_graph and mode == "pipelined")
        out = []
        for i in range(n):
            nxt = batches[i + 1] if (mode == "pipelined" and i + 1 < n and i != 6) else None   # one bubble at i == 6
            out.append(step(batches[i], next_data=nxt).clone())
        res[mode] = (torch.stack(out).cpu(), model._flat.params.clone(), float(model._flat.step))
    assert res["plain"][2] == res["pipelined"][2] == n
    assert torch.allclose(res["pipelined"][0], res["plain"][0], rtol=1e-4, atol=0)
    assert rel(res["pipelined"][1], res["plain"][1]) < 1e-3      # reduction-order noise through Adam, see above


def test_widened_vae_inference_with_overlap_add(dev):
    """BASELINE.json configs[4]: widened VAE (segment_length 4096, n_units 4096, latent 256) inference -
    frames of a wav at hop 512 -> encode -> latent -> decode -> overlap-add resynthesis - against the fp64 oracle
    (bf16 tolerance), with a ragged frame count (not a multiple of the 128-row tile)."""
    from rawvae.model import VAE
    from rawaudiovae_kelsey_b200 import ops
    from oracle import rawvae_oracle as O
    S, H, L, hop = 4096, 4096, 256, 512
    gen = torch.Generator().manual_seed(11)
    n = (600 - 1) * hop + S - 37                               # 600 frames after the reference's zero padding
    audio = (torch.rand(n, generator=gen) * 2 - 1)
    frames_ref = torch.from_numpy(O.audio_dataset_frames(audio.numpy(), S, hop))
    N = frames_ref.shape[0]
    assert N == O.audio_dataset_len(n, S, hop) == 600
    torch.manual_seed(0)
    model = VAE(S, H, L).to(dev).eval()
    p64 = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    frames, _, _ = ops.frame_gather(audio.to(dev), N, hop, S)
    assert torch.equal(frames.cpu(), frames_ref)               # framing is bit-exact
    mu, lv = model.encode(frames)
    eps = torch.randn(N, L, generator=gen)
    z = model.reparameterize(mu, lv, eps=eps.to(dev))
    xh = model.decode(z)
    act = O.forward(p64, frames_ref.double(), eps.double())
    assert rel(mu, act["mu"]) < BF16_TOL and rel(lv, act["logvar"]) < BF16_TOL
    assert rel(z, act["z"]) < BF16_TOL
    assert rel(xh, act["x_hat"]) < BF16_TOL
    # resynthesis: overlap-add of the decoded frames vs the oracle's OLA of the oracle's frames; and the identity
    # ola(frames(x)) == zero-padded x that pins the operation (SURVEY.md 8c)
    ola = ops.overlap_add(xh, hop)
    ola_ref = torch.from_numpy(O.resynth_overlap_add(act["x_hat"].float().numpy(), hop))
    assert ola.shape == ola_ref.shape and rel(ola, ola_ref) < BF16_TOL
    ident = ops.overlap_add(frames, hop).cpu()
    padded = torch.from_numpy(O.pad_to_multiple(audio.numpy(), hop))
    assert torch.allclose(ident[: padded.numel()], padded, atol=1e-6)


def _needs_experiments():
    from rawaudiovae_kelsey_b200 import _lib
    if not _lib.load().rvae_build_experiments():
        pytest.skip("measured-and-rejected path: only in builds with RVAE_EXPERIMENTS=1")


def test_chained_forward_launch_equals_separate_kernels(dev, monkeypatch):
    _needs_experiments()
    """RVAE_FUSE_FORWARD=1 runs fc1 -> head -> fc3 -> fc4/loss as ONE persistent launch whose tiles wait for the
    row blocks they consume (tile-level dependency counters). Same arithmetic, same operands: losses and weights
    match the four separate launches up to the reduction-order noise of the loss / bias-gradient atomics."""
    from rawvae.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, B, n = 512, 768, 128, 1300, 6          # 11 row blocks (ragged), several column blocks per layer
    gen = torch.Generator().manual_seed(21)
    x = (torch.rand(n, B, S, generator=gen) * 2 - 1).to(dev)
    eps = torch.randn(n, B, L, generator=gen).to(dev)
    res = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("RVAE_FUSE_FORWARD", mode)     # read when the plan is created
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        opt = Adam(model.parameters(), lr=1e-3)
        step = FusedTrainStep(model, opt, 1e-3, ring=8)
        losses = [float(step(x[i], eps=eps[i])) for i in range(n)]
        res[mode] = (torch.tensor(losses), model._flat.params.clone())
    assert torch.allclose(res["1"][0], res["0"][0], rtol=1e-4, atol=0)
    assert rel(res["1"][1], res["0"][1]) < 1e-3


@pytest.mark.parametrize("shape", [(512, 768, 128, 1300), (1024, 2048, 256, 768)])
def test_fused_latent_epilogue_matches_latent_kernel(dev, monkeypatch, shape):
    _needs_experiments()
    """RVAE_FUSE_LATENT=1 computes d_ml = [dz + c mu | dz eps sigma / 2 + c (sigma^2 - 1) / 2] and db2 in the epilogue
    of the latent dgrad GEMM (no split-K dz round trip, no latent backward kernel). Same formulas on the same
    operands as the kernel path: losses, weights and Adam moments agree up to accumulation-order noise. Ragged rows
    (B % 256 != 0) and a latent width below the tile width are covered by the first shape."""
    from rawvae.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, B = shape
    n = 4
    gen = torch.Generator().manual_seed(23)
    x = (torch.rand(n, B, S, generator=gen) * 2 - 1).to(dev)
    eps = torch.randn(n, B, L, generator=gen).to(dev)
    res = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("RVAE_FUSE_LATENT", mode)      # read when the plan is created
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        opt = Adam(model.parameters(), lr=1e-3)
        step = FusedTrainStep(model, opt, 1e-2, ring=8)   # a KL weight large enough for its gradient to matter
        losses = [float(step(x[0], eps=eps[0]))]
        # after the first step exp_avg = (1 - beta1) * gradient: compared per tensor, so that the 2L bias gradients
        # the epilogue sums itself are not drowned by the weight matrices
        flat = model._flat
        m1 = {name: flat.view(flat.exp_avg, name).clone() for name in flat.offsets}
        losses += [float(step(x[i], eps=eps[i])) for i in range(1, n)]
        res[mode] = (torch.tensor(losses), flat.params.clone(), m1)
    assert torch.allclose(res["1"][0], res["0"][0], rtol=1e-4, atol=0)
    for name, m in res["1"][2].items():
        assert rel(m, res["0"][2][name]) < 5e-3, name    # (a dropped row / column block would show as O(0.1 .. 1))
    # (Adam turns the accumulation-order noise of near-zero gradients into +-lr steps: measured 1.4e-3)
    assert rel(res["1"][1], res["0"][1]) < 5e-3


def test_alternating_batch_sizes_share_one_plan(dev, monkeypatch):
    """A plan serves every batch size up to its capacity (a ragged last batch of an epoch), but holds ONE set of
    fused-launch tile schedules: other batch sizes must fall back to separate launches instead of running the
    owner's schedule. Reference: the same steps with fused launches disabled."""
    from rawvae.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L = 512, 768, 128
    sizes = [1536, 700, 1536, 1024, 1536]
    gen = torch.Generator().manual_seed(29)
    xs = [(torch.rand(b, S, generator=gen) * 2 - 1).to(dev) for b in sizes]
    es = [torch.randn(b, L, generator=gen).to(dev) for b in sizes]
    res = {}
    for pairs in ("default", "0"):
        if pairs == "0":
            monkeypatch.setenv("RVAE_DUAL_PAIRS", "0")    # no fused launches at all
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        opt = Adam(model.parameters(), lr=1e-3)
        step = FusedTrainStep(model, opt, 1e-3, ring=8)
        losses = [float(step(x, eps=e)) for x, e in zip(xs, es)]
        res[pairs] = (torch.tensor(losses), model._flat.params.clone())
    assert torch.allclose(res["default"][0], res["0"][0], rtol=1e-4, atol=0)
    assert rel(res["default"][1], res["0"][1]) < 2e-3   # (a stale schedule drops tiles: O(1) after the third step)


def _write_wav_folder(root, n_files, seconds, sr, seed):
    from scipy.io import wavfile
    from oracle.rawvae_oracle import synth_wav
    rng = np.random.default_rng(seed)
    root.mkdir(parents=True, exist_ok=True)
    for i in range(n_files):
        x = synth_wav(rng, int(seconds * sr), sr)
        wavfile.write(root / f"clip{i}.wav", sr, np.round(x * 32767).astype(np.int16))


def _trainer_ini(path, datapath, *, batch, extra_training):
    path.write_text(f"""[audio]
sampling_rate = 44100
hop_length = 128
segment_length = 1024

[dataset]
datapath = {datapath}
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
batch_size = {batch}
loss_reduction = mean
{extra_training}

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
""")


@pytest.mark.parametrize("which", ["epoch", "stream"])
def test_drop_in_trainers_produce_reference_artefacts(dev, tmp_path, which):
    """train.py / train_iterable.py drop-ins (train.py:94-307, train_iterable.py:95-329) on a tiny synthetic wav
    folder: same workspace tree, and a checkpoint whose state_dict has the reference's keys / shapes (so it loads
    into the reference VAE, tutorial.ipynb:292-297) plus a torch.optim.Adam-format optimizer state."""
    from rawaudiovae_kelsey_b200 import trainer
    data = tmp_path / "data"
    _write_wav_folder(data / "audio", 3, 1.5, 44100, 1)
    _write_wav_folder(data / "test_audio", 1, 0.5, 44100, 2)
    ini = tmp_path / "cfg.ini"
    if which == "epoch":
        _trainer_ini(ini, data, batch=512, extra_training="epochs = 3\nsave_best_model_after = 1\ncheckpoint_interval = 2")
        rc = trainer.run_epoch_trainer(["--config", str(ini)])
    else:
        _trainer_ini(ini, data, batch=256,
                     extra_training="epochs = 1\ntotal_num_frames = 2560\ncheckpoint_interval = 4\nlog_interval = 2")
        rc = trainer.run_stream_trainer(["--config", str(ini)])
    assert rc in (0, None)
    runs = sorted((data / "unit-test").glob("run-*"))
    assert len(runs) == 1
    run = runs[0]
    assert (run / "config.ini").exists() and (run / "model" / "last_model.pt").exists()
    ckpts = sorted((run / "model" / "checkpoints").glob("ckpt_*"))
    assert ckpts, "no checkpoint written"
    state = torch.load(ckpts[-1], map_location="cpu", weights_only=False)
    sd = state["state_dict"]
    shapes = {"fc1.weight": (256, 1024), "fc1.bias": (256,), "fc21.weight": (64, 256), "fc21.bias": (64,),
              "fc22.weight": (64, 256), "fc22.bias": (64,), "fc3.weight": (256, 64), "fc3.bias": (256,),
              "fc4.weight": (1024, 256), "fc4.bias": (1024,)}
    assert {k: tuple(v.shape) for k, v in sd.items()} == shapes
    assert all(v.dtype == torch.float32 and torch.isfinite(v).all() for v in sd.values())
    opt = state["optimizer"]
    assert len(opt["state"]) == 10 and sorted(opt["state"][0]) == ["exp_avg", "exp_avg_sq", "step"]
    assert float(opt["state"][0]["step"]) > 0
    assert (run / "audio_logs" / "test_original.wav").exists()


def test_cpu_tensors_fail_loudly(dev):
    from rawvae.model import VAE, loss_function
    from rawaudiovae_kelsey_b200._lib import RvaeError
    m = VAE(128, 128, 64)
    with pytest.raises(RvaeError):
        m(torch.zeros(4, 128))                 # CPU model + CPU input: no fallback
    m = m.to(dev)
    with pytest.raises(RvaeError):
        m(torch.zeros(4, 128))                 # CPU input on a CUDA model
    with pytest.raises(RvaeError):
        loss_function(torch.zeros(4, 128), torch.zeros(4, 128), torch.zeros(4, 64), torch.zeros(4, 64), 1e-4, 128)


def test_inference_api_encode_reparameterize_decode(dev, small):
    """tutorial.ipynb pattern: encode -> lerp of (mu, logvar) in float64 -> reparameterize -> decode -> view(-1)."""
    from oracle import rawvae_oracle as O
    model = make_model(small, "init", dev, "fp32").eval()
    S, H, L, B, _ = (int(v) for v in small["meta"])
    x = torch.from_numpy(small["x"]).to(dev)
    with torch.no_grad():
        mu, lv = model.encode(x)
        assert rel(mu, small["mu"]) < FP32_TOL and rel(lv, small["logvar"]) < FP32_TOL
        a = 0.25
        mu_i = (1 - a) * mu[: B // 2].double() + a * mu[B // 2:].double()
        lv_i = (1 - a) * lv[: B // 2].double() + a * lv[B // 2:].double()
        eps = torch.randn(B // 2, L, device=dev)
        z = model.reparameterize(mu_i, lv_i, eps=eps)
        assert z.dtype == torch.float64
        assert rel(z, mu_i + eps.double() * torch.exp(0.5 * lv_i)) < 1e-6
        z2 = model.reparameterize(mu_i, lv_i)                  # internal Philox noise
        assert z2.shape == z.shape and not torch.equal(z2, z)
        xh = model.decode(z.float())
        p = {k: torch.from_numpy(small["init/" + k]).double() for k in O.PARAM_NAMES}
        zc = z.cpu().double()
        ref = torch.tanh(torch.clamp_min(zc @ p["fc3.weight"].T + p["fc3.bias"], 0) @ p["fc4.weight"].T + p["fc4.bias"])
        assert rel(xh, ref) < FP32_TOL
        assert xh.view(-1).numel() == (B // 2) * S
        x1d = model(x[0])[0]                                   # 1-D [S] input, as export-onnx.ipynb feeds
        assert x1d.shape == (1, S)


def test_checkpoint_roundtrip_with_reference_format(dev, small, tmp_path):
    """ckpt dict {state_dict, optimizer} (train_iterable.py:222-226) and whole-module pickles reload; the
    state_dict is plain fp32 tensors with the reference's keys/shapes."""
    from rawvae.model import VAE, loss_function
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, B, _ = (int(v) for v in small["meta"])
    model = make_model(small, "init", dev, "bf16")
    opt = Adam(model.parameters(), lr=1e-3)
    x = torch.from_numpy(small["x"]).to(dev)
    xh, mu, lv = model(x)
    loss_function(xh, x, mu, lv, 1e-4, S).backward()
    opt.step()
    state = {"batch_id": 1, "state_dict": model.state_dict(), "optimizer": opt.state_dict()}
    torch.save(state, tmp_path / "ckpt_00001")
    torch.save(model, tmp_path / "last_model.pt")
    ck = torch.load(tmp_path / "ckpt_00001", weights_only=False)
    assert list(ck["state_dict"].keys()) == [k for k, _ in model.named_parameters()]
    assert ck["state_dict"]["fc21.weight"].shape == (L, H) and ck["state_dict"]["fc21.weight"].dtype == torch.float32
    assert len(ck["optimizer"]["state"]) == 10 and ck["optimizer"]["param_groups"][0]["params"] == list(range(10))
    m2 = VAE(S, H, L).to(dev)
    m2.load_state_dict(ck["state_dict"])
    o2 = Adam(m2.parameters(), lr=1e-3)
    o2.load_state_dict(ck["optimizer"])
    eps = torch.randn(B, L, device=dev)
    a = model(x, eps=eps)[0]
    b = m2(x, eps=eps)[0]
    assert torch.equal(a, b)
    m3 = torch.load(tmp_path / "last_model.pt", weights_only=False)
    assert torch.equal(m3(x, eps=eps)[0], a)
    assert float(o2.state_dict()["state"][0]["step"]) == 1.0


@pytest.mark.parametrize("pcm16", [False, True])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_frames_read_in_place_equal_gathered_frames(dev, monkeypatch, precision, pcm16):
    """SURVEY.md 2c K-F1 / VERDICT r1 missing #6: a RUN of consecutive frames (IterableAudioDataset's stream,
    rawvae/dataset.py:61-69) is never materialised - the run's sample span is converted to bf16 once and fc1's A
    operand, the MSE side input and the fc1 weight gradient read frame i at row pitch hop through overlapping-row TMA
    tensor maps. Same operands, same tiles => the outputs equal the gather path's: activations bit for bit, sums that
    go through atomics to reassociation noise. Ragged batch (not a multiple of the 128-row tile), a run that starts
    mid-buffer and ends in the zero-padded tail, fp32 and PCM16 sources, eager / pipelined / graph-replayed steps."""
    from rawvae.model import VAE, FusedTrainStep, FrameBatch
    from rawaudiovae_kelsey_b200 import model as M
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, hop, B, first = 256, 320, 64, 64, 500, 37
    gen = torch.Generator().manual_seed(17)
    n_samples = (first + B - 1) * hop + S - 29               # the last frame reaches 29 samples past the buffer
    audio = (torch.rand(n_samples, generator=gen) * 2 - 1)
    audio = torch.round(audio * 32768).clamp_(-32768, 32767).to(torch.int16).to(dev) if pcm16 else audio.to(dev)
    eps = torch.randn(B, L, generator=gen).to(dev)

    def run(span_on):
        monkeypatch.setattr(M, "_SPAN_ON", span_on)
        torch.manual_seed(0)
        model = VAE(S, H, L, precision=precision).to(dev)
        fb = FrameBatch(audio, B, hop, S, first_frame=first)
        assert fb.span == span_on
        with torch.no_grad():
            xh, mu, lv = model(fb, eps=eps)
        plan = model._plan_for(B)
        assert plan.pitch == (hop if span_on else 0)
        step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-3), 1e-3, keep_grads=True)
        loss = step(fb, eps=eps).clone()
        return xh.clone(), mu.clone(), lv.clone(), loss, model._flat.grads.clone(), model._flat.params.clone()

    a, b = run(True), run(False)
    for k in range(3):
        assert torch.equal(a[k], b[k]), ("xhat", "mu", "logvar")[k]
    assert torch.allclose(a[3], b[3], rtol=1e-5, atol=0)
    assert rel(a[4], b[4]) < 1e-5 and rel(a[5], b[5]) < 1e-6
    # the materialised frames are the reference's (zero padded tail included)
    fr = FrameBatch(audio, B, hop, S, first_frame=first).materialize().cpu()
    a_cpu = audio.cpu().float() / (32768.0 if pcm16 else 1.0)
    a_pad = torch.cat([a_cpu, torch.zeros(64)])
    assert torch.equal(fr[-1], a_pad[(first + B - 1) * hop:(first + B - 1) * hop + S]) and torch.equal(fr[0], a_pad[first * hop:first * hop + S])

    if precision == "fp32" or pcm16:
        return
    # a stream of runs through the pipelined, graph-replayed step (first frame read from device memory on replay)
    starts = [5, 700, 333, 41, 1200, 64, 900, 2, 512, 77]
    long_audio = (torch.rand((1300 + B) * hop + S, generator=gen) * 2 - 1).to(dev)
    res = {}
    for span_on in (True, False):
        monkeypatch.setattr(M, "_SPAN_ON", span_on)
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        model.eps_seed = 5
        step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-3), 1e-3, ring=16, graph=True)
        fbs = [FrameBatch(long_audio, B, hop, S, first_frame=s) for s in starts]
        out = [step(fbs[i], next_data=fbs[i + 1] if i + 1 < len(fbs) else None).clone() for i in range(len(fbs))]
        if span_on:
            assert step.stats["replays"] >= 4, step.stats
        res[span_on] = (torch.stack(out).cpu(), model._flat.params.clone())
    assert torch.allclose(res[True][0], res[False][0], rtol=1e-4, atol=0)
    assert rel(res[True][1], res[False][1]) < 1e-3


def test_per_kernel_timing_mode_runs_the_same_step(dev):
    """bench.py's roofline attribution (rvae_plan_enable_timing): the step's own launches - the fused dgrad + weight
    gradient launches of backward stages 0 and 2 included, booked on the dgrad's slot with the flops of both problems -
    run one at a time between CUDA events. The step computes the same thing as the untimed step."""
    from rawvae.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, B = 1024, 2048, 256, 8192      # default.ini at the bench's batch: the shapes whose stages fuse
    gen = torch.Generator().manual_seed(3)
    x = (torch.rand(B, S, generator=gen) * 2 - 1).to(dev)
    eps = torch.randn(B, L, generator=gen).to(dev)
    res = {}
    for timed in (False, True):
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-3), 1e-3)
        plan = model._plan_for(B)
        plan.enable_timing(timed)
        losses = [step(x, eps=eps).clone() for _ in range(3)]
        torch.cuda.synchronize()
        if timed:
            tm = plan.read_timing()
            plan.enable_timing(False)
            assert tm["B4d"][1] == 3 and tm["B2d"][1] == 3 and tm["B3d"][1] == 3 and tm["B3w"][1] == 3 and tm["B1w"][1] == 3
            assert tm["B4w"][1] == 0 and tm["B2w"][1] == 0, "stages 0 and 2 run as ONE fused launch each"
            assert tm["B4d"][2] == 2.0 * B * H * S * 2 and tm["B2d"][2] == 2.0 * B * H * 2 * L * 2    # both problems' flops
            assert all(tm[k][0] > 0 for k in ("F1", "F2", "F3", "F4_out", "B4d", "B3d", "B3w", "B2d", "B1w", "adam", "latent_bwd"))
        res[timed] = (torch.stack(losses).cpu(), model._flat.params.clone())
    assert torch.allclose(res[True][0], res[False][0], rtol=1e-4, atol=0)
    assert rel(res[True][1], res[False][1]) < 2e-3      # reduction-order noise (split-K reduce-adds) through 3 Adam steps


@pytest.mark.parametrize("use_graph", [False, True])
def test_adam_kernel_equals_torch_adam_on_the_implementations_own_gradients(dev, use_graph):
    """VERDICT r1 weak 4: the end-to-end weight tolerances after a few steps (1e-3 / 1e-2) are wider than the
    activation / gradient tolerances because Adam's normalised update m / (sqrt(v) + eps) turns reassociation noise in
    near-zero gradient entries into O(lr) differences - NOT because the Adam kernel is loose. Isolate it: feed
    torch.optim.Adam (the reference's optimizer, train.py:163) the very gradients the fused step produced and compare
    parameters and both moments after 5 steps at 1e-6 - the kernel itself (torch's lerp / addcmul / sqrt / div order,
    fp64 bias corrections, bf16 shadow refresh) is exact to fp32 rounding. Also through CUDA-graph replays."""
    from rawvae.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    S, H, L, B, n = 256, 320, 64, 512, 5
    gen = torch.Generator().manual_seed(21)
    xs = [(torch.rand(B, S, generator=gen) * 2 - 1).to(dev) for _ in range(n)]
    torch.manual_seed(0)
    model = VAE(S, H, L).to(dev)
    model.eps_seed = 9
    opt = Adam(model.parameters(), lr=1e-3)
    step = FusedTrainStep(model, opt, 1e-3, keep_grads=True, graph=use_graph)
    flat = model._ensure_flat()
    ref_p = flat.params.detach().clone().requires_grad_(True)
    ref_opt = torch.optim.Adam([ref_p], lr=1e-3)
    for i in range(n):
        step(xs[i])
        torch.cuda.synchronize()
        ref_p.grad = flat.grads.detach().clone()           # the gradients this step's kernels produced
        ref_opt.step()
        st = ref_opt.state[ref_p]
        assert rel(flat.params, ref_p.detach()) < 1e-6, i
        assert rel(flat.exp_avg, st["exp_avg"]) < 1e-6 and rel(flat.exp_avg_sq, st["exp_avg_sq"]) < 1e-6, i
        assert torch.equal(flat.shadow_hi.float(), flat.params.to(torch.bfloat16).float()), "bf16 shadow = rn(params)"
    assert float(flat.step) == n == int(st["step"])
    if use_graph:
        assert step.stats["replays"] >= 2, step.stats
