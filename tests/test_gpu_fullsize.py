"""GPU parity tests at the sizes BASELINE.json names (-m gpu): the sm_100a path against the fp64 oracle ELEMENTWISE at
B = 8192 (default.ini) and B = 4096 (kelsey_iterable.ini), through the drop-in API route and through the route the
benchmark times (FusedTrainStep, CUDA-graph replay, background prefetch, in-library Philox noise); the Philox noise
itself; and data parallelism on real GPUs (2 ranks, skipped on a single-GPU box).

Tolerances are BASELINE.json's: fp32 mode <= 1e-4 relative, bf16 mode <= 2e-2 relative."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from test_gpu_parity import BF16_TOL, FP32_TOL, gated_reference, rel

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
S, H, L = 1024, 2048, 256            # default.ini:5,18-19
HOP, KL_BETA, LR = 128, 1e-4, 1e-4   # default.ini:4,20,26

# Gate flips allowed between the implementation's ReLU masks and the fp64 reference's (gated_reference already
# asserts every flip lies within tol * rms of zero): a pre-activation lands in that band with probability ~0.8 tol
# and flips in at most half of those cases.
MAX_FLIP_FRACTION = {"bf16": 0.4 * BF16_TOL, "fp32": 0.4 * FP32_TOL}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _corpus(dev, seconds=40.0, seed=3):
    from oracle.rawvae_oracle import synth_wav
    rng = np.random.default_rng(seed)
    wav = np.concatenate([synth_wav(rng, int(seconds * 44100 / 4)) for _ in range(4)])
    return torch.from_numpy(wav).to(dev)


def _p64(model):
    return {k: v.detach().double().cpu() for k, v in model.state_dict().items()}


def _check_against_oracle(model, p64, x, eps, got, precision, tol, B):
    """got: dict with optional x_hat / mu / logvar / loss and the 10 gradients, all from the implementation."""
    from oracle import rawvae_oracle as O
    act, gref, flips = gated_reference(model, p64, x, eps, KL_BETA, tol)
    units = B * 2 * H
    assert flips <= MAX_FLIP_FRACTION[precision] * units, f"{flips} gate flips of {units} units"
    for name in ("x_hat", "mu", "logvar"):
        if name in got:
            assert rel(got[name], act[name]) < tol, name
    ref_loss = float(O.loss_function(act["x_hat"], act["x"], act["mu"], act["logvar"], KL_BETA, S))
    assert abs(got["loss"] - ref_loss) < tol * ref_loss, (got["loss"], ref_loss)
    for k in O.PARAM_NAMES:
        assert rel(got["grads"][k], gref[k]) < tol, f"gradient {k}: {rel(got['grads'][k], gref[k]):.3e}"
    return flips


# ------------------------------------------------------------------------------------------------ API route, real sizes
@pytest.mark.parametrize("B", [8192, 4096])
@pytest.mark.parametrize("precision,tol", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_api_route_elementwise_vs_oracle_at_config_size(dev, precision, tol, B):
    """model(x) -> loss_function -> backward at S/H/L = 1024/2048/256, B = 8192 (BASELINE.json configs[1]) and 4096
    (configs[3], kelsey_iterable.ini:26): x_hat, mu, logvar, the loss and all 10 gradients elementwise (relative L2)
    against oracle.forward / oracle.backward in fp64 (rawvae/model.py:19-46)."""
    from rawvae.model import VAE, loss_function
    torch.manual_seed(0)
    model = VAE(S, H, L, precision=precision).to(dev)
    gen = torch.Generator().manual_seed(11)
    x = torch.rand(B, S, generator=gen) * 2 - 1
    eps = torch.randn(B, L, generator=gen)
    xh, mu, lv = model(x.to(dev), eps=eps.to(dev))
    loss = loss_function(xh, x.to(dev), mu, lv, KL_BETA, S)
    loss.backward()
    got = {"x_hat": xh, "mu": mu, "logvar": lv, "loss": loss.item(),
           "grads": {k: p.grad for k, p in model.named_parameters()}}
    _check_against_oracle(model, _p64(model), x, eps, got, precision, tol, B)


# ------------------------------------------------------------------------------------------------ the timed route
@pytest.mark.parametrize("B,sequential", [(8192, False), (4096, True)])
@pytest.mark.parametrize("precision,tol", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_graph_replay_prefetch_philox_step_vs_oracle(dev, precision, tol, B, sequential):
    """The path bench.py times - FusedTrainStep(graph=True), next batch prefetched on the background stream, noise
    from the in-library Philox generator, fused dgrad+wgrad launches - checked against the ORACLE (not against the
    eager CUDA path): the 7th step is a graph replay; its loss, mu, logvar and all 10 gradients are compared with
    oracle.forward / backward in fp64 evaluated at the weights before that step, on the frames the step gathered and
    the noise it drew (read back from the plan). B = 8192 random gather (default.ini); B = 4096 consecutive frames
    of a stream (kelsey_iterable.ini)."""
    from rawvae.model import VAE, FusedTrainStep, FrameBatch
    from rawaudiovae_kelsey_b200.optim import Adam
    from oracle import rawvae_oracle as O
    torch.manual_seed(0)
    model = VAE(S, H, L, precision=precision).to(dev)
    model.eps_seed = 5
    opt = Adam(model.parameters(), lr=LR)
    step = FusedTrainStep(model, opt, KL_BETA, graph=True, keep_grads=True)
    audio = _corpus(dev)
    n_frames = (audio.numel() - S) // HOP + 1
    n = 8
    gen = torch.Generator().manual_seed(21)
    if sequential:
        batches = [FrameBatch(audio, B, HOP, S, first_frame=int(torch.randint(0, n_frames - B, (1,), generator=gen)))
                   for _ in range(n + 1)]
    else:
        idx = torch.randint(0, n_frames, (n + 1, B), generator=gen).to(dev)
        batches = [FrameBatch(audio, B, HOP, S, frame_idx=idx[i]) for i in range(n + 1)]
    for i in range(n - 2):
        step(batches[i], next_data=batches[i + 1])
    assert step.stats["captures"] == 2 and step.stats["eager"] == 2 and step.steady >= 2, step.stats
    torch.cuda.synchronize()
    p64 = _p64(model)
    before = dict(step.stats)
    loss = step(batches[n - 2], next_data=batches[n - 1])
    torch.cuda.synchronize()
    assert step.stats["replays"] == before["replays"] + 1 and step.stats["captures"] == before["captures"]
    plan = model._plan_for(B)
    x = batches[n - 2].materialize().cpu()
    eps = plan.latent("eps").clone().cpu()
    flat = model._flat
    got = {"mu": plan.latent("mu").clone(), "logvar": plan.latent("logvar").clone(), "loss": float(loss),
           "grads": {k: flat.view(flat.grads, k).clone() for k in O.PARAM_NAMES}}
    # plan activations (ReLU gates) are still those of this step: the background prefetch only touched the alternate set
    _check_against_oracle(model, p64, x, eps, got, precision, tol, B)
    # and the noise really is N(0,1)-like and fresh per step
    assert abs(float(eps.mean())) < 5e-3 and abs(float(eps.std()) - 1.0) < 5e-3


# ------------------------------------------------------------------------------------------------ Philox noise
def test_philox_noise_distribution_and_independence(dev):
    """randn_kernel (replaces torch.randn_like, rawvae/model.py:25): 8 M samples - mean, variance, skewness, kurtosis,
    a Kolmogorov-Smirnov test against N(0,1); no correlation across offsets (steps) or seeds; and the data-parallel
    contract: a rank's rows drawn with elem_base = row0 * L are bit-identical to that slice of the single-process
    tensor, so shards are disjoint pieces of one stream (never the same noise on two ranks)."""
    from scipy import stats
    from rawaudiovae_kelsey_b200 import ops
    n = 8 * 1024 * 1024
    a = ops.randn((n,), seed=1234, offset=7, device=dev)
    x = a.double().cpu().numpy()
    assert abs(x.mean()) < 4.0 / np.sqrt(n)                       # 4 sigma
    assert abs(x.var() - 1.0) < 4.0 * np.sqrt(2.0 / n)
    assert abs(stats.skew(x)) < 4.0 * np.sqrt(6.0 / n)
    assert abs(stats.kurtosis(x)) < 4.0 * np.sqrt(24.0 / n)
    assert np.abs(x).max() > 4.5 and np.abs(x).max() < 7.0        # tails exist and are not absurd
    ks = stats.kstest(x[:: 8], "norm")
    assert ks.pvalue > 1e-3, ks
    # independence across the step offset, the seed, and neighbouring elements
    b = ops.randn((n,), seed=1234, offset=8, device=dev).double().cpu().numpy()
    c = ops.randn((n,), seed=1235, offset=7, device=dev).double().cpu().numpy()
    for other in (b, c, np.roll(x, 1), np.roll(x, 4), np.roll(x, 256)):
        assert abs(np.corrcoef(x, other)[0, 1]) < 4.0 / np.sqrt(n)
    # data-parallel shards: rows [r0, r1) of a [B, L] tensor
    B, Lz = 8192, 256
    full = ops.randn((B, Lz), seed=99, offset=3, device=dev)
    for r0, r1 in ((0, 1024), (1024, 2048), (4096, 8192), (8191, 8192)):
        part = ops.randn((r1 - r0, Lz), seed=99, offset=3, device=dev, elem_base=r0 * Lz)
        assert torch.equal(part, full[r0:r1])
    assert not torch.equal(full[:4096], full[4096:])


# ------------------------------------------------------------------------------------------------ inference API (N3)
def test_inference_api_interpolation_pattern_vs_oracle(dev):
    """tutorial.ipynb:456-470 (raw_to_z_dist), :496-510 (global alpha), :905-932 (per-frame float64 alpha from
    interp1d) through the product API: encode_audio -> lerp_latents -> decode_latents -> resynthesize, and the chained
    interpolate(); against the oracle in fp64 with injected eps."""
    from scipy import interpolate as sp_interpolate
    from rawvae.model import VAE
    from rawaudiovae_kelsey_b200 import inference as inf
    from oracle import rawvae_oracle as O
    torch.manual_seed(0)
    S_, H_, L_ = 1024, 2048, 256
    model = VAE(S_, H_, L_, precision="fp32").to(dev).eval()
    p64 = _p64(model)
    rng = np.random.default_rng(5)
    wav_a = O.synth_wav(rng, 200 * S_ + 300)       # ragged tail: TestDataset zero-pads to a multiple of S
    wav_b = O.synth_wav(rng, 200 * S_ + 300)
    mu_a, lv_a = inf.encode_audio(model, wav_a, batch_size=64)      # TestDataset framing (hop = S), as cell 13-14
    mu_b, lv_b = inf.encode_audio(model, wav_b, batch_size=64)
    N = mu_a.shape[0]
    assert N == 201 and mu_b.shape == (N, L_)
    fr_a = torch.from_numpy(O.test_dataset_frames(wav_a, S_)).double()
    ref_a = O.forward(p64, fr_a, torch.zeros(N, L_, dtype=torch.float64))
    assert rel(mu_a, ref_a["mu"]) < FP32_TOL and rel(lv_a, ref_a["logvar"]) < FP32_TOL
    # per-frame alpha exactly as the notebook builds it (cell 37)
    interpolation = 0.5 + 0.5 * np.sin(np.linspace(0, 6 * np.pi, 50))
    f_stretch = sp_interpolate.interp1d(np.arange(0, len(interpolation)), interpolation)
    alpha = f_stretch(np.linspace(0.0, len(interpolation) - 1, N))                # float64 [N]
    eps = torch.randn(N, L_, generator=torch.Generator().manual_seed(2))
    al = torch.from_numpy(alpha).to(dev)
    z, mu_i, lv_i = inf.lerp_latents(mu_a, lv_a, mu_b, lv_b, al, eps=eps.to(dev), return_dist=True)
    a64 = torch.from_numpy(alpha)[:, None]
    mu_ref = mu_a.double().cpu() * (1 - a64) + mu_b.double().cpu() * a64
    lv_ref = lv_a.double().cpu() * (1 - a64) + lv_b.double().cpu() * a64
    z_ref = mu_ref + eps.double() * torch.exp(0.5 * lv_ref)
    assert rel(mu_i, mu_ref) < 1e-6 and rel(lv_i, lv_ref) < 1e-6 and rel(z, z_ref) < 1e-6
    x_ref = torch.tanh(torch.relu(z_ref @ p64["fc3.weight"].T + p64["fc3.bias"]) @ p64["fc4.weight"].T + p64["fc4.bias"])
    frames = inf.decode_latents(model, z, batch_size=64)
    assert rel(frames, x_ref) < FP32_TOL
    audio = inf.resynthesize(frames, mode="concat")
    assert audio.shape == (N * S_,) and torch.equal(audio, frames.reshape(-1))   # tutorial.ipynb:543,932
    # one chained call: lerp -> reparameterize -> decode (z goes straight into fc3's operand), same result
    chained = inf.interpolate(model, mu_a, lv_a, mu_b, lv_b, al, eps=eps.to(dev), batch_size=96)
    assert rel(chained, x_ref) < FP32_TOL
    # global alpha sweep of cell 16: 6 x N frames
    sweep = inf.interpolate(model, mu_a, lv_a, mu_b, lv_b, [0.0, 0.2, 0.4, 0.6, 0.8, 1.0], eps=eps.to(dev))
    assert sweep.shape == (6 * N, S_)
    z0 = mu_a.double().cpu() + eps.double() * torch.exp(0.5 * lv_a.double().cpu())
    x0 = torch.tanh(torch.relu(z0 @ p64["fc3.weight"].T + p64["fc3.bias"]) @ p64["fc4.weight"].T + p64["fc4.bias"])
    assert rel(sweep[:N], x0) < FP32_TOL
    # overlap-add resynthesis of hop-128 frames (the "extensions" cells use AudioDataset framing): identity on x itself
    fr = torch.from_numpy(O.audio_dataset_frames(wav_a, S_, HOP)).to(dev)
    ola = inf.resynthesize(fr, mode="ola", hop=HOP)
    assert torch.allclose(ola.cpu(), torch.from_numpy(O.pad_to_multiple(wav_a, HOP)), atol=1e-6)
    # streamed reconstruction (encode -> reparameterize -> decode -> overlap-add, batch by batch with a carry of the last
    # S/hop - 1 decoded frames) == everything at once; ragged last batch, batch smaller than the carry included
    mu_h, lv_h = inf.encode_audio(model, wav_a, hop=HOP)
    Nh = mu_h.shape[0]
    eps_h = torch.randn(Nh, L_, generator=torch.Generator().manual_seed(3)).to(dev)
    whole = inf.resynthesize(inf.decode_latents(model, inf.lerp_latents(mu_h, lv_h, mu_h, lv_h, 0.0, eps=eps_h)),
                             mode="ola", hop=HOP)
    for bs in (Nh, 500, 37, 5):
        streamed = inf.reconstruct_audio(model, wav_a, hop=HOP, batch_size=bs, eps=eps_h)
        assert streamed.shape == whole.shape and float((streamed - whole).abs().max()) < 2e-5, bs
    rec = inf.reconstruct_audio(model, wav_a, batch_size=64, sample=False)          # TestDataset framing + concat
    mean_path = inf.decode_latents(model, mu_a)
    assert rec.shape == (N * S_,) and float((rec - mean_path.reshape(-1)).abs().max()) < 2e-5
    # bf16 mode within its tolerance too
    model.set_precision("bf16")
    assert rel(inf.interpolate(model, mu_a, lv_a, mu_b, lv_b, al, eps=eps.to(dev)), x_ref) < BF16_TOL


# ------------------------------------------------------------------------------------------------ whole-module pickle
def test_whole_module_pickle_loads_without_this_package_and_stays_small(dev, tmp_path):
    """torch.save(model, last_model.pt) of a CUDA model that has trained (train_iterable.py:314-315): the file holds
    the parameters only (not gradients / Adam moments / bf16 shadows) and unpickles in a process where `rawvae.model`
    is a stub with nothing but a VAE class - i.e. where this package does not exist (the reference's own notebook)."""
    from rawvae.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    torch.manual_seed(0)
    model = VAE(256, 320, 64).to(dev)
    step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-3), 1e-3)
    step(torch.rand(128, 256, device=dev) * 2 - 1)
    torch.cuda.synchronize()
    path = tmp_path / "last_model.pt"
    torch.save(model, path)
    n_param_bytes = 4 * sum(p.numel() for p in model.parameters())
    assert path.stat().st_size < 1.1 * n_param_bytes + 65536, (path.stat().st_size, n_param_bytes)
    stub = tmp_path / "stub" / "rawvae"
    stub.mkdir(parents=True)
    (stub / "__init__.py").write_text("")
    (stub / "model.py").write_text("import torch.nn as nn\nclass VAE(nn.Module):\n    pass\n")
    code = ("import sys, torch; sys.path.insert(0, sys.argv[1]);\n"
            "m = torch.load(sys.argv[2], map_location='cpu', weights_only=False)\n"
            "assert type(m).__module__ == 'rawvae.model' and 'rawaudiovae_kelsey_b200' not in sys.modules\n"
            "sd = m.state_dict(); assert sorted(sd) == sorted(['fc1.weight','fc1.bias','fc21.weight','fc21.bias',"
            "'fc22.weight','fc22.bias','fc3.weight','fc3.bias','fc4.weight','fc4.bias']), sorted(sd)\n"
            "print(float(sd['fc1.weight'].double().sum()))\n")
    res = subprocess.run([sys.executable, "-c", code, str(tmp_path / "stub"), str(path)], capture_output=True, text=True,
                         cwd=str(tmp_path), env={k: v for k, v in os.environ.items() if k != "PYTHONPATH"})
    assert res.returncode == 0, res.stderr
    assert abs(float(res.stdout.strip()) - float(model.fc1.weight.double().sum())) < 1e-6


# ------------------------------------------------------------------------------------------------ data parallel, 2 GPUs
def _torchrun(n, script, *args, env=None, timeout=600):
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(script), *map(str, args)]
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run(cmd, capture_output=True, text=True, cwd=str(ROOT), env=e, timeout=timeout)


def _need_gpus(n):
    if torch.cuda.device_count() < n:
        pytest.skip(f"needs {n} GPUs; logs of the multi-GPU runs are under profiles/")


@pytest.mark.parametrize("world,backend", [(2, "p2p"), (2, "nvls"), (4, "auto"), (8, "auto"), (8, "p2p")])
def test_data_parallel_step_equals_single_process_step_on_gpus(world, backend):
    """SURVEY.md section 4 'distributed' row on hardware: W ranks, each with its shard of a global batch, through
    DataParallelTrainStep (the library's own all-reduce kernel, per-bucket Adam) == the single-process
    FusedTrainStep on the concatenated batch - losses, weights, Adam moments, 3 steps, unequal shards - and the
    replicas stay bit-identical. Also with in-library noise: the ranks' Philox draws are the single-process draw.
    Both exchange flavours: peer loads + posted peer writes over CUDA-IPC mappings ("p2p"), and the in-switch reduction
    over an NVLS multicast mapping (multimem.ld_reduce / multimem.st, "nvls"; "auto" picks it from 3 ranks up)."""
    _need_gpus(world)
    res = _torchrun(world, ROOT / "tools" / "dp_check.py", env={"RVAE_DP_BACKEND": backend})
    assert res.returncode == 0 and "DP CHECK PASSED" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
    assert "philox shards match the single-process draw: True" in res.stdout, res.stdout[-3000:]
    want_mc = backend == "nvls" or (backend == "auto" and world >= 3)
    assert f"multicast exchange: {want_mc}" in res.stdout, res.stdout[-3000:]


def test_stream_trainer_under_torchrun_survives_a_slow_checkpoint(tmp_path):
    """train_iterable.py under torchrun, 2 ranks, with rank 0's checkpoint block made slower (3 s) than the old 2 s
    all-reduce trap: the run completes, the ranks end with identical weights, the artefacts exist."""
    _need_gpus(2)
    from test_gpu_parity import _trainer_ini, _write_wav_folder
    data = tmp_path / "data"
    _write_wav_folder(data / "audio", 3, 2.0, 44100, 1)
    _write_wav_folder(data / "test_audio", 1, 0.5, 44100, 2)
    ini = tmp_path / "s.ini"
    _trainer_ini(ini, data, batch=512,
                 extra_training="epochs = 1\ntotal_num_frames = 6144\ncheckpoint_interval = 4\nlog_interval = 4")
    res = _torchrun(2, ROOT / "tools" / "dp_trainer_check.py", "--config", ini, "--slow", 3, "--dump", tmp_path / "w")
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    run = next((data / "unit-test").glob("run-*"))
    assert (run / "model" / "last_model.pt").exists() and (run / "model" / "checkpoints" / "ckpt_00012").exists()
    w0, w1 = torch.load(tmp_path / "w.rank0"), torch.load(tmp_path / "w.rank1")
    assert torch.equal(w0, w1)
