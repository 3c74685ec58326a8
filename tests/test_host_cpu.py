"""CPU-only tests (-m "not gpu"): host logic, the drop-in dataset classes against the reference's golden frames,
the C-ABI library (loads, exports every symbol of include/rvae_b200.h, rejects bad arguments without a GPU), and
the data-parallel exchange on world_size-2 gloo."""
import ctypes
import os
import re
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent


# ------------------------------------------------------------------------------------------------ C ABI
def test_library_builds_loads_and_exports_every_declared_symbol():
    from rawaudiovae_kelsey_b200 import _lib
    lib = _lib.load()
    header = (ROOT / "include" / "rvae_b200.h").read_text()
    declared = sorted(set(re.findall(r"\b(rvae_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 45
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/rvae_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
    assert lib.rvae_abi_version() == _lib.ABI_VERSION == 5


def test_param_layout_matches_reference_parameter_count():
    from rawaudiovae_kelsey_b200 import _lib
    lib = _lib.load()
    lay = _lib.Layout()
    assert lib.rvae_param_layout(1024, 2048, 256, ctypes.byref(lay)) == 0
    assert lay.total == 5772800                       # default.ini VAE (SURVEY.md 8a a1)
    assert lay.w2 - lay.w1 == 2048 * 1024 and lay.b1 == 1024 * 2048 * 2 + 2 * 256 * 2048 + 2048 * 256
    assert lib.rvae_param_layout(4096, 4096, 256, ctypes.byref(lay)) == 0
    assert lay.total == 36712960                      # widened inference config (SURVEY.md 8a a13)
    # unsupported shapes fail loudly with a message, not silently
    rc = lib.rvae_param_layout(1000, 2048, 256, ctypes.byref(lay))
    assert rc == 2 and b"multiples of 64" in lib.rvae_last_error()


def test_no_gpu_means_loud_failure_not_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from rawaudiovae_kelsey_b200 import _lib, ops
    from rawvae.model import VAE, loss_function
    with pytest.raises(_lib.RvaeError):
        ops.ctx()
    m = VAE(128, 128, 64)
    with pytest.raises(_lib.RvaeError):
        m(torch.zeros(2, 128))
    with pytest.raises(_lib.RvaeError):
        loss_function(torch.zeros(2, 128), torch.zeros(2, 128), torch.zeros(2, 64), torch.zeros(2, 64), 1e-4, 128)
    out = ctypes.c_void_p()
    assert _lib.load().rvae_ctx_create(0, ctypes.byref(out)) != 0


def test_product_path_never_imports_the_oracle():
    for pkg in ("rawaudiovae_kelsey_b200", "rawvae"):
        for f in (ROOT / pkg).rglob("*.py"):
            src = f.read_text()
            assert "oracle" not in re.sub(r'""".*?"""', "", src, flags=re.S).replace("# ", ""), f
    for f in ("train.py", "train_iterable.py"):
        if (ROOT / f).exists():
            assert "import oracle" not in (ROOT / f).read_text() and "from oracle" not in (ROOT / f).read_text()


# ------------------------------------------------------------------------------------------------ model surface
def test_vae_surface_matches_reference():
    from rawvae.model import VAE
    torch.manual_seed(0)
    m = VAE(1024, 2048, 256)
    assert (m.segment_length, m.n_units, m.latent_dim) == (1024, 2048, 256)
    assert [k for k, _ in m.named_parameters()] == ["fc1.weight", "fc1.bias", "fc21.weight", "fc21.bias",
                                                    "fc22.weight", "fc22.bias", "fc3.weight", "fc3.bias",
                                                    "fc4.weight", "fc4.bias"]
    assert m.fc21.weight.shape == (256, 2048) and m.fc4.weight.shape == (1024, 2048)
    assert sum(p.numel() for p in m.parameters()) == 5772800
    from oracle.rawvae_oracle import init_params
    ref = init_params(1024, 2048, 256, seed=0)
    for k, p in m.named_parameters():
        assert torch.equal(p.detach(), ref[k]), k       # same default init stream as the reference
    assert VAE.__module__ == "rawvae.model"


def test_reference_forward_traces_and_matches_the_oracle():
    """SURVEY.md 8f N4 (export-onnx.ipynb:361-362): the ctypes kernels are invisible to a tracer, so forward() routes to
    reference_forward - plain torch ops on the same parameters - while traced / exported. Its values equal the
    oracle's, and torch.jit.trace(model, torch.randn(1024)) (the notebook's 1-D example input; the TorchScript ONNX
    exporter traces the same way) yields a graph with the reference's outputs. No onnx runtime exists in this image."""
    from rawvae.model import VAE
    from oracle import rawvae_oracle as O
    torch.manual_seed(0)
    m = VAE(1024, 256, 64)
    p = {k: v.detach().double() for k, v in m.state_dict().items()}
    gen = torch.Generator().manual_seed(3)
    x = torch.rand(5, 1024, generator=gen) * 2 - 1
    eps = torch.randn(5, 64, generator=gen)
    xh, mu, lv = m.reference_forward(x, eps)
    act = O.forward(p, x.double(), eps.double())
    for got, want in ((xh, act["x_hat"]), (mu, act["mu"]), (lv, act["logvar"])):
        assert float((got.double() - want).norm() / want.norm()) < 1e-6
    one = torch.randn(1024, generator=gen)
    traced = torch.jit.trace(m, (one, torch.zeros(1, 64)), check_trace=False)     # forward() itself, on CPU
    t_xh, t_mu, t_lv = traced(one, torch.zeros(1, 64))
    r_xh, r_mu, r_lv = m.reference_forward(one, torch.zeros(1, 64))
    assert t_xh.shape == (1, 1024) and torch.allclose(t_xh, r_xh) and torch.allclose(t_mu, r_mu)
    ops = {n.kind() for n in traced.graph.nodes()} | {n.kind() for n in traced.inlined_graph.nodes()}
    assert any("tanh" in k for k in ops) and any("linear" in k or "addmm" in k for k in ops), ops
    with pytest.raises(Exception):
        m(one)        # an ordinary (untraced) call on CPU still fails loudly: no CPU fallback


def test_vae_pickles_like_a_plain_module(tmp_path):
    from rawvae.model import VAE
    m = VAE(128, 192, 64)
    torch.save(m, tmp_path / "best_model.pt")
    m2 = torch.load(tmp_path / "best_model.pt", weights_only=False)
    assert type(m2).__module__ == "rawvae.model"
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k
    for private in ("_flat", "_plans"):
        assert private not in m.__getstate__()


# ------------------------------------------------------------------------------------------------ datasets
@pytest.fixture(scope="module")
def ds(golden_dir):
    return np.load(golden_dir / "dataset.npz")


@pytest.mark.parametrize("n", [22087, 1024, 1025, 2048, 1151, 1152])
def test_dataset_classes_bit_exact_vs_reference(ds, n):
    from rawvae.dataset import AudioDataset, TestDataset, ToTensor
    audio = ds[f"audio_{n}"]
    a = AudioDataset(audio, 1024, 44100, 128, transform=ToTensor())
    t = TestDataset(audio, 1024, 44100, transform=ToTensor())
    assert [len(a), len(t)] == [int(v) for v in ds[f"audio_len_{n}"]]
    got = np.stack([a[int(i)].numpy() for i in ds[f"audio_idx_{n}"]])
    np.testing.assert_array_equal(got, ds[f"audio_frames_{n}"])
    np.testing.assert_array_equal(np.stack([t[i].numpy() for i in range(len(t))]), ds[f"test_frames_{n}"])
    assert isinstance(a[0], torch.Tensor) and a[0].dtype == torch.float32
    with pytest.raises(ValueError):
        AudioDataset(audio, 1000, 44100, 128)


def test_iterable_dataset_stream_bit_exact_vs_reference(ds, tmp_path):
    import scipy.io.wavfile as wavfile
    from torch.utils.data import DataLoader
    from rawvae.dataset import IterableAudioDataset
    order = [str(s) for s in ds["stream_order"]]
    for name in order:
        wavfile.write(str(tmp_path / name), 44100, ds["stream_pcm_" + name])
    it = IterableAudioDataset(tmp_path, 44100, 128, torch.float32, torch.device("cpu"), shuffle=False)
    assert it.num_files == 3
    it.audio_file_list = [tmp_path / n for n in order]
    batches = []
    for b in DataLoader(it, batch_size=50, shuffle=False):        # train_iterable.py:151
        batches.append(b)
        if len(batches) == 3:
            break
    np.testing.assert_array_equal(torch.cat(batches).numpy(), ds["stream_frames"])
    it.shuffle = True
    assert sorted(p.name for p in it.shuffled_data_list) == sorted(order)


def test_sampler_permutation_reproduces_dataloader_shuffle():
    from torch.utils.data import DataLoader
    from rawaudiovae_kelsey_b200.dataset import sampler_permutation, shard_bounds
    n, bs = 1000, 64
    torch.manual_seed(123)
    ref = torch.cat([b for b in DataLoader(torch.arange(n), batch_size=bs, shuffle=True)])
    torch.manual_seed(123)
    got = sampler_permutation(n)
    assert torch.equal(ref, got)                                   # bit-exact frame indices (train.py:134)
    for world in (1, 2, 3, 8):
        cover = []
        for r in range(world):
            lo, hi = shard_bounds(61, r, world)
            cover += list(range(lo, hi))
        assert cover == list(range(61))


def test_init_test_audio_artifacts(tmp_path):
    import scipy.io.wavfile as wavfile
    from rawvae.tests import init_test_audio
    from rawaudiovae_kelsey_b200 import audio_io
    ta = tmp_path / "test_audio"
    ta.mkdir()
    rng = np.random.default_rng(0)
    pcm = np.clip(np.round(rng.standard_normal(3000) * 2000), -32768, 32767).astype(np.int16)
    wavfile.write(str(ta / "t0.wav"), 44100, pcm)
    work = tmp_path / "run-000"
    work.mkdir()
    dsx, logdir = init_test_audio(work, "test_audio", ta, 44100, 1024)
    assert logdir == work / "audio_logs" and (logdir / "test_audio.txt").exists()
    assert (logdir / "test_original.wav").exists()
    assert len(dsx) == 3 and dsx[0].dtype == torch.float32             # 3000 -> padded 3072 = 3 frames
    back, sr = audio_io.load_mono(logdir / "test_original.wav", 44100)
    np.testing.assert_array_equal(back, pcm.astype(np.float32) / 32768.0)


# ------------------------------------------------------------------------------------------------ data parallel (gloo)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, B, ret):
    sys.path.insert(0, str(ROOT))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from oracle import rawvae_oracle as O
    from rawaudiovae_kelsey_b200 import dist as rdist
    from rawaudiovae_kelsey_b200.dataset import shard_bounds
    r, w, _ = rdist.init_from_env("gloo")
    assert (r, w) == (rank, world)
    S, H, L, beta = 128, 192, 64, 1e-2
    p = {k: v.double() for k, v in O.init_params(S, H, L, seed=0).items()}
    gen = torch.Generator().manual_seed(1)
    x = (torch.rand(B, S, generator=gen) * 2 - 1).double()
    eps = torch.randn(B, L, generator=gen).double()
    lo, hi = shard_bounds(B, rank, world)
    act = O.forward(p, x[lo:hi], eps[lo:hi])
    # normalise the local loss by the GLOBAL batch (what rvae_plan_set_global_batch does): scale = local/global
    scale = (hi - lo) / B
    g = O.backward(p, act, beta, grad_out=scale)
    flat = torch.cat([g[k].flatten() for k in O.PARAM_NAMES])
    buckets = [flat[: flat.numel() // 2], flat[flat.numel() // 2:]]
    for wk in rdist.allreduce_buckets(buckets):
        wk.wait()
    if rank == 0:
        act_full = O.forward(p, x, eps)
        gf = O.backward(p, act_full, beta)
        ref = torch.cat([gf[k].flatten() for k in O.PARAM_NAMES])
        ret.put(float((flat - ref).norm() / ref.norm()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("B", [64, 61])
def test_data_parallel_sum_allreduce_equals_single_process_gradient(B):
    """world_size 2 over gloo: sharded gradients with global-batch loss normalisation, SUM all-reduced in buckets,
    equal the single-process gradient of the concatenated batch - equal and unequal shards."""
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, B, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert ret.get(timeout=5) < 1e-12


def test_ingest_ring_logic_with_mocked_cuda(tmp_path, monkeypatch):
    """GpuFrameStream's host logic (file placement in a ring smaller than the corpus, region reuse, batches that
    straddle files, resampled / stereo files, rank sharding) without a GPU: CUDA streams and events are mocked, the
    ring lives in host memory and frames are gathered with numpy from the (first_frame | frame_idx) descriptors. Every
    frame equals the CPU IterableAudioDataset stream's; with the one-batch lookahead of the trainers, too."""
    from itertools import islice
    from test_gpu_parity import _write_mixed_corpus
    from rawaudiovae_kelsey_b200 import dataset as D
    from rawaudiovae_kelsey_b200.trainer import _with_next

    class Ev:
        def record(self, *_): pass
    class St:
        def wait_event(self, *_): pass
        def __enter__(self): return self
        def __exit__(self, *a): return False
    monkeypatch.setattr(torch.cuda, "Stream", lambda **k: St())
    monkeypatch.setattr(torch.cuda, "Event", lambda **k: Ev())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: St())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: s)

    class HostRingStream(D.GpuFrameStream):
        def __init__(self, ds, bs, **kw):
            self.ds, self.batch_size, self.device = ds, bs, torch.device("cpu")
            self.pcm16, self.rank, self.world = False, kw.get("rank", 0), kw.get("world", 1)
            self.dtype, self.esize, self.capacity, self.lookahead = torch.float32, 4, kw["capacity"], 2
            self.ring, self.stats = None, {"files_uploaded": 0, "bytes_uploaded": 0, "resident_hits": 0, "ring_wraps": 0}
        def _decode(self, path):
            a = self.ds.load_file(path).contiguous()
            return a, a                      # (staged view, its staging buffer)
        def _release(self, buf, ev):
            pass

    def gather(fb):
        idx = fb.frame_idx.numpy() if fb.frame_idx is not None else fb.first_frame + np.arange(fb.n_frames)
        a = fb.audio.numpy()
        return np.stack([a[i * fb.hop: i * fb.hop + fb.segment_length].copy() for i in idx])

    names = _write_mixed_corpus(tmp_path)
    ds = D.IterableAudioDataset(tmp_path, 44100, 128, torch.float32, "cpu", shuffle=False)
    ds.audio_file_list = names
    B, n_batches = 32, 200
    want = torch.stack(list(islice(iter(ds), B * n_batches))).numpy()
    total = sum(ds.load_file(f).numel() for f in names)
    cap = int(0.4 * total) // 1024 * 1024
    st = HostRingStream(ds, B, capacity=cap)
    got = np.concatenate([gather(fb) for fb in islice(iter(st), n_batches)])     # gather BEFORE asking for the next batch
    np.testing.assert_array_equal(got, want)
    assert st.stats["ring_wraps"] >= 3 and st.stats["files_uploaded"] > len(names) and st.ring.numel() == cap
    # trainer-style lookahead: batch k is gathered only after batch k + 1 has been requested
    st = HostRingStream(ds, B, capacity=cap)
    got = np.concatenate([gather(cur) for cur, nxt in _with_next(islice(iter(st), n_batches))])
    np.testing.assert_array_equal(got, want)
    # everything resident: one upload per file, later cycles are hits
    st = HostRingStream(ds, B, capacity=2 * total)
    got = np.concatenate([gather(fb) for fb in islice(iter(st), n_batches)])
    np.testing.assert_array_equal(got, want)
    assert st.stats["files_uploaded"] == len(names) and st.stats["resident_hits"] > len(names)
    # data parallel: the ranks' shards tile every global batch
    ranks = [iter(HostRingStream(ds, B, capacity=cap, rank=r, world=3)) for r in range(3)]
    for k in range(60):
        shards = [next(it) for it in ranks]
        rows = np.concatenate([gather(fb) for fb in shards])
        np.testing.assert_array_equal(rows, want[k * B:(k + 1) * B])
        assert [fb.global_row0 for fb in shards] == [0, 11, 22] and shards[0].global_batch == B
    # a ring that cannot hold a file next to its predecessor says so instead of corrupting a pending batch
    with pytest.raises(RuntimeError, match="too small|does not fit"):
        list(islice(iter(HostRingStream(ds, B, capacity=24 * 1024)), n_batches))


def test_trainer_lookahead_pairs():
    """trainer._with_next: (batch, next batch) pairs in order, None after the last - what lets a training step
    prefetch the next batch in the background (device-side analogue of the DataLoader's prefetch)."""
    from rawaudiovae_kelsey_b200.trainer import _with_next
    assert list(_with_next([])) == []
    assert list(_with_next([1])) == [(1, None)]
    assert list(_with_next(iter("abc"))) == [("a", "b"), ("b", "c"), ("c", None)]


def test_bench_data_generator_matches_the_tests_generator():
    """bench.py restates the SURVEY.md 8(d) wav generator so that its GPU arm imports nothing from oracle/; the two
    stay bit-identical. And no module of the product package imports the oracle."""
    import importlib
    import re
    from pathlib import Path
    from oracle.rawvae_oracle import synth_wav
    bench = importlib.import_module("bench")
    a = bench.synth_wav(np.random.default_rng(7), 5000)
    b = synth_wav(np.random.default_rng(7), 5000)
    assert a.dtype == np.float32 and np.array_equal(a, b)
    root = Path(bench.__file__).resolve().parent
    for f in list((root / "rawaudiovae_kelsey_b200").glob("*.py")) + list((root / "rawvae").glob("*.py")):
        assert not re.search(r"^\s*(from|import)\s+oracle", f.read_text(), re.M), f


def test_bench_dump_outputs_files(tmp_path):
    """bench.py --dump-outputs at the benchmark's dimensions: the loss, every parameter in full and the same seeded
    sample of both Adam moments on every call, all float32, 64 MB at most."""
    import importlib
    from rawvae.model import VAE
    bench = importlib.import_module("bench")
    torch.manual_seed(0)
    model = VAE(bench.S, bench.H, bench.L)
    opt = torch.optim.Adam(model.parameters(), lr=bench.LR)
    for p in model.parameters():
        p.grad = torch.randn_like(p)
    opt.step()
    loss = torch.tensor(0.25)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), model, opt, loss)
    names = ["loss", "exp_avg.sample", "exp_avg_sq.sample"] + [k for k, _ in model.named_parameters()]
    assert sorted(f.name for f in (tmp_path / "a").iterdir()) == sorted(n + ".npy" for n in names)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 * 2 ** 20
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in names}
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["loss"] == np.float32(0.25)
    for k, p in model.named_parameters():
        assert np.array_equal(got[k], p.detach().numpy()), k
    for key in ("exp_avg", "exp_avg_sq"):
        full = torch.cat([opt.state[p][key].flatten() for p in model.parameters()]).numpy()
        assert got[key + ".sample"].size == bench.MOMENT_SAMPLE and np.isin(got[key + ".sample"], full).all()
        assert np.array_equal(got[key + ".sample"], np.load(tmp_path / "b" / (key + ".sample.npy")))


def test_pcm16_passthrough_view_equals_the_decoded_file(tmp_path):
    """The streaming ingest copies 16-bit PCM files into pinned memory as they are (audio_io.open_pcm16); the int16
    values it hands to the GPU are exactly the ones the float decode (int16 / 32768, what torchaudio.load returns,
    rawvae/dataset.py:47) rounds back to. Stereo files keep their channel layout ([samples, channels]: channel 0 is
    column 0, :54-55); non-PCM16 files are refused (None) so the caller falls back to the float path."""
    import scipy.io.wavfile as wavfile
    from rawaudiovae_kelsey_b200 import audio_io
    rng = np.random.default_rng(3)
    mono = rng.integers(-32768, 32767, 5000, dtype=np.int16)
    stereo = rng.integers(-32768, 32767, (4000, 2), dtype=np.int16)
    wavfile.write(tmp_path / "m.wav", 44100, mono)
    wavfile.write(tmp_path / "s.wav", 48000, stereo)
    wavfile.write(tmp_path / "f.wav", 44100, rng.standard_normal(100).astype(np.float32))
    d, sr = audio_io.open_pcm16(tmp_path / "m.wav")
    x, sr2 = audio_io.load_wav_channels(tmp_path / "m.wav")
    assert sr == sr2 == 44100 and d.dtype == np.int16 and np.array_equal(np.asarray(d), mono)
    assert np.array_equal(np.asarray(d).astype(np.float32) / 32768.0, x[0])
    d, sr = audio_io.open_pcm16(tmp_path / "s.wav")
    x, _ = audio_io.load_wav_channels(tmp_path / "s.wav")
    assert sr == 48000 and d.shape == (4000, 2) and np.array_equal(np.asarray(d[:, 0]).astype(np.float32) / 32768.0, x[0])
    assert audio_io.open_pcm16(tmp_path / "f.wav")[0] is None


def test_resident_audio_keeps_16_bit_pcm_content_as_int16_only_when_lossless(monkeypatch):
    """dataset.resident_audio: a float corpus decoded from 16-bit PCM (k / 32768) is held as int16 - the framing kernel's
    int16 * (1 / 32768) gives back every float exactly - anything else stays float32; RVAE_PCM16_RESIDENT=0 disables."""
    from rawaudiovae_kelsey_b200 import dataset as D
    rng = np.random.default_rng(5)
    pcm = rng.integers(-32768, 32768, 10000, dtype=np.int64).astype(np.int16)
    pcm[:2] = (-32768, 32767)
    as_float = pcm.astype(np.float32) / 32768.0
    t = D.resident_audio(as_float, "cpu")
    assert t.dtype == torch.int16 and np.array_equal(t.numpy(), pcm)
    assert np.array_equal(t.numpy().astype(np.float32) * np.float32(1.0 / 32768.0), as_float)     # what the kernel computes
    assert D.resident_audio(pcm, "cpu").dtype == torch.int16
    noisy = as_float.copy()
    noisy[1234] += 1e-6                                   # one sample off the 16-bit grid: not lossless any more
    assert D.resident_audio(noisy, "cpu").dtype == torch.float32
    assert D.resident_audio(np.array([1.0, 0.0], dtype=np.float32), "cpu").dtype == torch.float32   # +1.0 = 32768 / 32768
    assert D.resident_audio(rng.standard_normal(100), "cpu").dtype == torch.float32
    monkeypatch.setenv("RVAE_PCM16_RESIDENT", "0")
    assert D.resident_audio(as_float, "cpu").dtype == torch.float32
