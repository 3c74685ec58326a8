"""Cost of a scheduled training step: steady-state CUDA-graph steps of FusedTrainStep at B = 8192 and the default dims
(1024, 2048, 256), bf16, with the constant schedule against a cosine learning rate with warm-up plus a cyclical KL
weight. The two runs alternate within one process, `--rounds` times, each timing `--steps` replayed steps with CUDA
events after a warm-up that captures the graph.

    python tools/schedule_perf.py [--steps 200] [--rounds 3] [--out DIR]

Prints one JSON object (GPU name and power limit included); --out DIR also writes it to DIR/r3_schedule_perf.json."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from padded_dims_perf import gpu_info  # noqa: E402

B, DIMS = 8192, (1024, 2048, 256)


def make_step(schedule, dev):
    from rawaudiovae_kelsey_b200.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    torch.manual_seed(0)
    model = VAE(*DIMS, precision="bf16").to(dev)
    model.eps_seed = 1
    opt = Adam(model.parameters(), lr=1e-4)
    return FusedTrainStep(model, opt, kl_beta=1e-4, graph=True, schedule=schedule)


def timed_steps(step, x, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        step(x)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    from rawaudiovae_kelsey_b200.schedule import Schedule
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    x = torch.from_numpy(np.random.default_rng(0).uniform(-0.5, 0.5, (B, DIMS[0])).astype(np.float32)).to(dev)
    total = 10 * args.steps * args.rounds
    runs = {"constant": make_step(None, dev),
            "cosine+cyclical": make_step(Schedule("cosine", 100, total, 1e-6, "cyclical", 0.0, 1, 4, 0.5), dev)}
    for step in runs.values():
        for _ in range(5):
            step(x)
    res = {k: [] for k in runs}
    for _ in range(args.rounds):
        for name, step in runs.items():
            start = step.stats["replays"]
            res[name].append(timed_steps(step, x, args.steps))
            assert step.stats["replays"] - start == args.steps   # every timed step was a graph replay
    out = {"gpu": gpu_info(), "batch": B, "dims": DIMS, "precision": "bf16", "steps_per_round": args.steps,
           "step_ms": res, "median_ms": {k: float(np.median(v)) for k, v in res.items()}}
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_schedule_perf.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
