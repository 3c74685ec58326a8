"""GPU parameter histograms (rvae_param_histogram, stats.ParamHistogramLogger) against TensorBoard's make_histogram:
exact counts / limits / min / max / num, fp64 moments to 1e-12, bitwise reproducibility, ordering against the
training step (CUDA graphs + prefetching), widened dims, and the trainers' event files."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytest.importorskip("tensorboard")
from torch.utils.tensorboard.summary import make_histogram  # noqa: E402

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(Path(__file__).resolve().parent))

pytestmark = pytest.mark.gpu

from rawaudiovae_kelsey_b200 import ops, stats  # noqa: E402

EDGES = np.asarray(stats.default_bins(), dtype=np.float64)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda", 0)


class _RawWriter:
    """Collects what add_histogram_raw receives."""

    def __init__(self):
        self.calls = []

    def add_histogram_raw(self, tag, global_step=None, walltime=None, **fields):
        self.calls.append((tag, global_step, fields))


def _check(fields, values: np.ndarray, what=""):
    """fields (add_histogram_raw kwargs) == make_histogram(values) exactly, moments to 1e-12 relative."""
    ref = make_histogram(values.astype(np.float64), EDGES)
    assert fields["bucket_limits"] == list(ref.bucket_limit), what
    assert fields["bucket_counts"] == list(ref.bucket), what
    assert fields["num"] == ref.num, what
    for k in ("min", "max"):
        a, b = fields[k], getattr(ref, k)
        assert (a == b) or (np.isnan(a) and np.isnan(b)), (what, k, a, b)
    # the moments are summed in another order than numpy's: 1e-12 relative to the sum of magnitudes (the sum of
    # values that cancel, e.g. +-1e20, has no relative accuracy of its own)
    v64 = values.astype(np.float64).ravel()
    scale = {"sum": np.abs(v64).sum(), "sum_squares": v64.dot(v64)}
    for k in ("sum", "sum_squares"):
        a, b = fields[k], getattr(ref, k)
        if np.isfinite(b):
            assert abs(a - b) <= 1e-12 * max(scale[k], 1e-300), (what, k, a, b)
        else:
            assert (a == b) or (np.isnan(a) and np.isnan(b)), (what, k, a, b)


def _hist(params, segs):
    offs = [o for o, _ in segs]
    lens = [n for _, n in segs]
    rec = ops.param_histogram(params, offs, lens, EDGES)
    lay = ops.histogram_record_layout(len(segs), EDGES.size)
    host = rec[:lay["bytes"]].cpu()
    r = ops.unpack_histogram_record(host, len(segs), EDGES.size)
    return rec, [stats.histogram_fields(r["counts"][i], EDGES, r["min"][i], r["max"][i], r["num"][i], r["sum"][i],
                                        r["sum_squares"][i]) for i in range(len(segs))]


def _model_segs(model):
    flat = model._ensure_flat()
    return flat, [(flat.offsets[n][0], p.numel()) for n, p in model.named_parameters()]


def _train(model, steps, B=512, graph=False, seed=0):
    from rawaudiovae_kelsey_b200.model import FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    g = torch.Generator(device="cpu").manual_seed(seed)
    S, hop = model.segment_length, 256
    audio = (torch.rand((B + 8) * hop + S, generator=g) * 2 - 1).to(model.fc1.weight.device)
    step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-3), 1e-4, graph=graph)
    for _ in range(steps):
        step(FrameBatch(audio, B, hop, S))
    torch.cuda.synchronize()


def test_default_dims_after_training_equal_make_histogram(dev):
    from rawaudiovae_kelsey_b200.model import VAE
    torch.manual_seed(0)
    model = VAE(1024, 2048, 256).to(dev)
    _train(model, 3)
    flat, segs = _model_segs(model)
    _, fields = _hist(flat.params, segs)
    for (name, p), f in zip(model.named_parameters(), fields):
        _check(f, p.detach().cpu().numpy(), name)


def _adversarial():
    e32 = EDGES.astype(np.float32)
    e32 = e32[np.isfinite(e32)]
    up, dn = np.nextafter(e32, np.float32(np.inf)), np.nextafter(e32, np.float32(-np.inf))
    rng = np.random.default_rng(3)
    fmax = np.finfo(np.float32).max
    return [
        np.concatenate([e32, up, dn, np.array([0.0, -0.0, 0.0], np.float32)]),
        np.array([1e-45, -1e-45, 1.1754942e-38, -1.1754942e-38, 3e-42, 0.0, 1e-12, -1e-12], np.float32),
        np.concatenate([np.array([fmax, -fmax, np.inf, -np.inf], np.float32),
                        rng.uniform(-1, 1, 999).astype(np.float32)]),
        np.concatenate([np.array([np.nan, 0.25, np.nan], np.float32), rng.normal(0, 3, 5000).astype(np.float32)]),
        np.full(70001, 0.0237, np.float32),
        np.zeros(2048, np.float32),
        (rng.standard_normal(40000) * 10.0 ** rng.uniform(-44, 37, 40000)).astype(np.float32),
    ]


def test_adversarial_values_equal_make_histogram(dev):
    parts = _adversarial()
    gap = 13   # segments need not be adjacent or aligned
    segs, chunks, off = [], [], 0
    for p in parts:
        chunks.append(np.full(gap, 7.0, np.float32))
        off += gap
        segs.append((off, p.size))
        chunks.append(p)
        off += p.size
    buf = torch.from_numpy(np.concatenate(chunks)).to(dev)
    _, fields = _hist(buf, segs)
    for i, (p, f) in enumerate(zip(parts, fields)):
        _check(f, p, f"segment {i}")


def test_repeated_calls_are_bitwise_identical(dev):
    from rawaudiovae_kelsey_b200.model import VAE
    torch.manual_seed(1)
    model = VAE(1024, 2048, 256).to(dev)
    flat, segs = _model_segs(model)
    lay = ops.histogram_record_layout(len(segs), EDGES.size)
    a, _ = _hist(flat.params, segs)
    a = a[:lay["bytes"]].clone()
    b, _ = _hist(flat.params, segs)
    assert torch.equal(a, b[:lay["bytes"]])


def test_bad_arguments_are_rejected(dev):
    from rawaudiovae_kelsey_b200._lib import RvaeError
    x = torch.zeros(100, device=dev)
    with pytest.raises(RvaeError):
        ops.param_histogram(x.cpu(), [0], [10], EDGES)
    with pytest.raises(RvaeError):
        ops.param_histogram(x, [95], [10], EDGES)
    with pytest.raises(RvaeError):
        ops.param_histogram(x, [0], [0], EDGES)
    with pytest.raises(RvaeError):
        ops.param_histogram(x, [0], [10], EDGES[::-1].copy())
    with pytest.raises(RvaeError):
        ops.param_histogram(x, [0], [10], np.linspace(-1, 1, 4096))
    with pytest.raises(RvaeError):
        ops.param_histogram(x, [0] * 17, [1] * 17, EDGES)


def test_records_follow_graph_replays_with_prefetch_without_host_sync(dev):
    """graph=True + next_data: record after step t and a clone of the parameters taken at the same point of the same
    stream agree for every t (the next step's background Adam must not overtake the record)."""
    from rawaudiovae_kelsey_b200.model import VAE, FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    torch.manual_seed(2)
    model = VAE(1024, 2048, 256).to(dev)
    B, S, hop, n = 1024, 1024, 128, 8
    g = torch.Generator(device="cpu").manual_seed(5)
    audio = (torch.rand((B * (n + 1)) * hop + S, generator=g) * 2 - 1).to(dev)
    batches = [FrameBatch(audio, B, hop, S, first_frame=i * B) for i in range(n + 1)]
    step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-3), 1e-4, graph=True)
    writer = _RawWriter()
    hist = stats.ParamHistogramLogger(model, writer, slots=n)
    clones = []
    for t in range(n):
        step(batches[t], next_data=batches[t + 1])
        hist.record(t)
        clones.append(model._flat.params.clone())
    hist.flush(wait=True)
    assert step.stats["replays"] >= 3, step.stats
    names = [nm for nm, _ in model.named_parameters()]
    assert len(writer.calls) == n * len(names)
    flat = model._flat
    for k, (tag, t, fields) in enumerate(writer.calls):
        assert tag == names[k % len(names)] and t == k // len(names)
        off, shape = flat.offsets[tag]
        vals = clones[t][off:off + int(np.prod(shape))].cpu().numpy()
        _check(fields, vals, f"{tag} @ {t}")
    assert not torch.equal(clones[0], clones[-1])


def test_widened_dims_counts_exact(dev):
    from rawaudiovae_kelsey_b200.model import VAE
    torch.manual_seed(4)
    model = VAE(4096, 4096, 256).to(dev)
    flat, segs = _model_segs(model)
    assert model.fc1.weight.numel() == 4096 * 4096
    _, fields = _hist(flat.params, segs)
    for (name, p), f in zip(model.named_parameters(), fields):
        _check(f, p.detach().cpu().numpy(), name)


def _events(run):
    # the legacy loader keeps histogram summaries as HistogramProto (EventFileLoader migrates them to tensors)
    from tensorboard.backend.event_processing.event_file_loader import LegacyEventFileLoader
    files = sorted((run / "logs").glob("events.out.tfevents.*"))
    hist, losses = {}, set()
    for f in files:
        for ev in LegacyEventFileLoader(str(f)).Load():
            for v in ev.summary.value:
                if v.HasField("histo"):
                    hist.setdefault(ev.step, {})[v.tag] = v.histo
                elif v.tag == "Loss/Batch":
                    losses.add(ev.step)
    return files, hist, sorted(losses)


def _corpus(tmp_path, seconds=1.5):
    from test_gpu_parity import _write_wav_folder
    data = tmp_path / "data"
    _write_wav_folder(data / "audio", 3, seconds, 44100, 1)
    _write_wav_folder(data / "test_audio", 1, 0.5, 44100, 2)
    return data


def test_stream_trainer_writes_every_batch_histograms_equal_to_final_checkpoint(dev, tmp_path):
    from test_gpu_parity import _trainer_ini
    from rawaudiovae_kelsey_b200 import trainer
    data = _corpus(tmp_path)
    ini = tmp_path / "s.ini"
    _trainer_ini(ini, data, batch=256, extra_training="epochs = 1\ntotal_num_frames = 2560\ncheckpoint_interval = 4\n"
                                                      "log_interval = 3\nhistogram_interval = 1")
    assert trainer.run_stream_trainer(["--config", str(ini)]) in (0, None)
    run = next((data / "unit-test").glob("run-*"))
    _, hist, batches = _events(run)
    names = ["fc1.weight", "fc1.bias", "fc21.weight", "fc21.bias", "fc22.weight", "fc22.bias", "fc3.weight",
             "fc3.bias", "fc4.weight", "fc4.bias"]
    assert len(batches) >= 5 and sorted(hist) == batches == list(range(len(batches)))
    assert all(sorted(h) == sorted(names) for h in hist.values())
    last = sorted((run / "model" / "checkpoints").glob("ckpt_*"))[-1]
    sd = torch.load(last, map_location="cpu", weights_only=False)["state_dict"]
    for name in names:
        h = hist[batches[-1]][name]
        ref = make_histogram(sd[name].numpy().astype(np.float64), EDGES)
        assert list(h.bucket_limit) == list(ref.bucket_limit) and list(h.bucket) == list(ref.bucket), name
        assert (h.min, h.max, h.num) == (ref.min, ref.max, ref.num), name
        assert abs(h.sum - ref.sum) <= 1e-12 * abs(ref.sum) and abs(h.sum_squares - ref.sum_squares) <= \
            1e-12 * ref.sum_squares, name


def test_epoch_trainer_writes_one_histogram_set_per_epoch(dev, tmp_path):
    from test_gpu_parity import _trainer_ini
    from rawaudiovae_kelsey_b200 import trainer
    data = _corpus(tmp_path)
    ini = tmp_path / "e.ini"
    _trainer_ini(ini, data, batch=512, extra_training="epochs = 2\nsave_best_model_after = 1\ncheckpoint_interval = 1")
    assert trainer.run_epoch_trainer(["--config", str(ini)]) in (0, None)
    run = next((data / "unit-test").glob("run-*"))
    _, hist, _ = _events(run)
    assert sorted(hist) == [0, 1] and all(len(h) == 10 for h in hist.values())
    sd = torch.load(run / "model" / "checkpoints" / "ckpt_00002", map_location="cpu", weights_only=False)["state_dict"]
    ref = make_histogram(sd["fc4.weight"].numpy().astype(np.float64), EDGES)
    assert list(hist[1]["fc4.weight"].bucket) == list(ref.bucket)


def test_stream_trainer_under_torchrun_histograms_on_rank0_only(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from test_gpu_fullsize import _torchrun
    from test_gpu_parity import _trainer_ini
    data = _corpus(tmp_path, 2.0)
    ini = tmp_path / "d.ini"
    _trainer_ini(ini, data, batch=512, extra_training="epochs = 1\ntotal_num_frames = 3072\ncheckpoint_interval = 4\n"
                                                      "log_interval = 2\nhistogram_interval = 1")
    res = _torchrun(2, ROOT / "tools" / "dp_trainer_check.py", "--config", ini, "--slow", 0)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    runs = list((data / "unit-test").glob("run-*"))
    assert len(runs) == 1   # only rank 0 has a workspace, hence the only event file
    files, hist, batches = _events(runs[0])
    assert len(files) == 1 and len(batches) >= 2 and sorted(hist) == batches
    assert all(len(h) == 10 for h in hist.values())
