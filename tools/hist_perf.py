"""python tools/hist_perf.py [--out DIR]

Cost of TensorBoard parameter histograms (rvae_param_histogram / stats.ParamHistogramLogger) on the GPU, printed and
(with --out) written to DIR/hist_perf.json, with the GPU name and power limit read in the same run:

  kernel    time of one record (memset + param_histogram_kernel) at the default (S=1024, H=2048, L=256) and widened
            (S=H=4096) dims, from CUDA events around a CUDA graph of 50 back-to-back records (parameters L2-warm
            when they fit the L2, as right after Adam) and of 50 records each preceded by a 256 MB L2-evicting write
            (cold; the write's own time, measured alone, is subtracted). Achieved bytes/s over the 4 B/parameter
            algorithmic traffic.
  step      steady-state FusedTrainStep(graph=True, next_data prefetching) step time with a record after every step
            (flushed every 64 steps into a null writer) vs no record, alternating A/B blocks.
  host      host time per histogram set of 10 parameters: the previous `writer.add_histogram(name, param, step)` loop
            (device sync, D2H copy, np.histogram) vs record + flush(wait=True), both into a real SummaryWriter.
  trainer   wall time of a short synthetic stream-trainer run at histogram_interval = 1, 64 and 0.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from rawaudiovae_kelsey_b200 import ops, stats  # noqa: E402
from rawaudiovae_kelsey_b200.model import VAE, FrameBatch, FusedTrainStep  # noqa: E402
from rawaudiovae_kelsey_b200.optim import Adam  # noqa: E402


class NullWriter:
    def add_histogram_raw(self, *a, **k):
        pass


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unavailable",
            "torch_name": torch.cuda.get_device_name(0)}


def graph_ms(fn, reps, iters=5):
    """Mean device ms per call of fn, captured `reps` times in one CUDA graph and replayed `iters` times."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / (iters * reps)


def kernel_times(dev):
    out = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    edges = np.asarray(stats.default_bins())
    for tag, (S, H, L) in (("default", (1024, 2048, 256)), ("widened", (4096, 4096, 256))):
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        flat = model._ensure_flat()
        offs = [flat.offsets[n][0] for n, _ in model.named_parameters()]
        lens = [p.numel() for _, p in model.named_parameters()]
        rec = torch.empty(ops.histogram_record_layout(len(offs), edges.size)["total"], dtype=torch.uint8, device=dev)
        n = sum(lens)
        rec_fn = lambda: ops.param_histogram(flat.params, offs, lens, edges, out=rec)
        warm = graph_ms(rec_fn, 50)
        flush_only = graph_ms(lambda: flush.fill_(1), 50)
        cold = graph_ms(lambda: (flush.fill_(1), rec_fn()), 50) - flush_only
        out[tag] = {"params": n, "param_bytes": 4 * n, "warm_us": warm * 1e3, "cold_us": cold * 1e3,
                    "warm_GBps": 4 * n / (warm * 1e-3) / 1e9, "cold_GBps": 4 * n / (cold * 1e-3) / 1e9,
                    "l2_warm_possible": 4 * n < 126e6}
        del model, flat
    return out


def step_overhead(dev, B, steps=256, blocks=3):
    torch.manual_seed(0)
    model = VAE(1024, 2048, 256).to(dev)
    step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-4), 1e-4, graph=True)
    hist = stats.ParamHistogramLogger(model, NullWriter())
    S, hop = 1024, 128
    n_b = 64
    audio = (torch.rand(B * n_b * hop // 8 + S + B * hop, device=dev) * 2 - 1)
    max_first = (audio.numel() - S) // hop - B
    batches = [FrameBatch(audio, B, hop, S, first_frame=(i * 7919 * 8) % max_first) for i in range(n_b)]

    def run(k, with_hist):
        for i in range(k):
            step(batches[i % n_b], next_data=batches[(i + 1) % n_b])
            if with_hist:
                hist.record(i)
                if i % 64 == 63:
                    hist.flush()
        hist.flush(wait=True)

    run(32, True)
    run(32, False)
    torch.cuda.synchronize()
    res = {"off": [], "on": []}
    for _ in range(blocks):
        for mode in ("off", "on"):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(steps, mode == "on")
            torch.cuda.synchronize()
            res[mode].append((time.perf_counter() - t0) / steps * 1e3)
    return {"batch": B, "steps_per_block": steps, "ms_per_step_off": res["off"], "ms_per_step_on": res["on"],
            "median_off": float(np.median(res["off"])), "median_on": float(np.median(res["on"])),
            "graph_stats": dict(step.stats)}


def host_per_set(dev, sets=10):
    from torch.utils.tensorboard import SummaryWriter
    torch.manual_seed(0)
    model = VAE(1024, 2048, 256).to(dev)
    model._ensure_flat()
    out = {}
    with tempfile.TemporaryDirectory() as d:
        w = SummaryWriter(log_dir=d)
        for name, p in model.named_parameters():   # warm-up of both paths
            w.add_histogram(name, p, 0)
        hist = stats.ParamHistogramLogger(model, w)
        hist.record(0)
        hist.flush(wait=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(sets):
            for name, p in model.named_parameters():
                w.add_histogram(name, p, s)
        out["old_add_histogram_ms"] = (time.perf_counter() - t0) / sets * 1e3
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(sets):
            hist.record(s)
            hist.flush(wait=True)
        out["gpu_record_flush_ms"] = (time.perf_counter() - t0) / sets * 1e3
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(sets):
            hist.record(s)
        torch.cuda.synchronize()
        out["record_only_ms"] = (time.perf_counter() - t0) / sets * 1e3
        hist.flush(wait=True)
        w.close()
    return out


def trainer_walls(tmp: Path):
    from test_gpu_parity import _write_wav_folder
    from rawaudiovae_kelsey_b200 import trainer
    data = tmp / "data"
    _write_wav_folder(data / "audio", 4, 20.0, 44100, 1)
    _write_wav_folder(data / "test_audio", 1, 0.5, 44100, 2)
    res = {}
    batches, batch = 256, 4096
    for interval in (1, 64, 0):
        ini = tmp / f"h{interval}.ini"
        ini.write_text(f"""[audio]
sampling_rate = 44100
hop_length = 128
segment_length = 1024
[dataset]
datapath = {data}
test_dataset = test_audio
generate_test = False
run_number = 0
workspace =
total_frames =
[VAE]
latent_dim = 256
n_units = 2048
kl_beta = 0.0001
[training]
learning_rate = 0.0001
batch_size = {batch}
total_num_frames = {batch * batches}
checkpoint_interval = 100000
log_interval = 64
histogram_interval = {interval}
[extra]
description = hist-{interval}
""")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        trainer.run_stream_trainer(["--config", str(ini)])
        torch.cuda.synchronize()
        res[f"interval_{interval}_s"] = time.perf_counter() - t0
    res["batches"], res["batch"] = batches, batch
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for hist_perf.json (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hist_perf.py measures on a CUDA device; none found")
    dev = torch.device("cuda", 0)
    out = {"gpu": gpu_info()}
    out["kernel"] = kernel_times(dev)
    print(json.dumps(out["kernel"], indent=1), flush=True)
    out["step"] = [step_overhead(dev, B) for B in (4096, 16384)]
    print(json.dumps(out["step"], indent=1), flush=True)
    out["host_per_set"] = host_per_set(dev)
    print(json.dumps(out["host_per_set"], indent=1), flush=True)
    with tempfile.TemporaryDirectory() as d:
        out["trainer_wall"] = trainer_walls(Path(d))
    print(json.dumps(out["trainer_wall"], indent=1), flush=True)
    out["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        Path(args.out, "hist_perf.json").write_text(json.dumps(out, indent=1))
    print(json.dumps(out["gpu"]))


if __name__ == "__main__":
    main()
