"""Cost of the exponential moving average (EMA) of the weights in the fused training step: steady-state CUDA-graph
steps of FusedTrainStep at B = 8192 and the default dims (1024, 2048, 256), bf16, with the EMA off and on, and the same
pair with gradient clipping on (max_grad_norm = 1.0). The four runs alternate within one process, `--rounds` times,
each timing `--steps` replayed steps with CUDA events after a warm-up that captures the graph. Also the HBM bytes per
parameter the step's Adam launches move, counted from what the kernel reads and writes.

With `--parent DIR` (a built checkout of the parent commit) it also runs `bench.py --gpus 1` in DIR and in this
checkout, alternating, `--bench-rounds` times: the EMA is off there, so the two must agree within their spread.

    python tools/ema_perf.py [--steps 200] [--rounds 3] [--parent DIR] [--bench-rounds 3] [--out DIR]

Prints one JSON object (GPU name and power limit included); --out DIR also writes it to DIR/r3_ema_perf.json."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from padded_dims_perf import gpu_info  # noqa: E402

B, DIMS = 8192, (1024, 2048, 256)
DECAY = 0.999


def make_step(ema_on, max_grad_norm, dev):
    from rawaudiovae_kelsey_b200.ema import ExponentialMovingAverage
    from rawaudiovae_kelsey_b200.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    torch.manual_seed(0)
    model = VAE(*DIMS, precision="bf16").to(dev)
    model.eps_seed = 1
    opt = Adam(model.parameters(), lr=1e-4)
    ema = ExponentialMovingAverage(model, DECAY) if ema_on else None
    return FusedTrainStep(model, opt, kl_beta=1e-4, graph=True, max_grad_norm=max_grad_norm, ema=ema)


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def adam_bytes_per_param(ema_on):
    """HBM bytes per parameter of the step's Adam launches (bf16 mode, gradients cleared by Adam): p, g, m, v read;
    p, m, v written; g cleared; the bf16 shadow written; with the EMA, e read and written."""
    return 4 * 4 + 3 * 4 + 4 + 2 + (8 if ema_on else 0)


def bench(tree, args):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.bench_steps), "--warmup",
           str(args.bench_warmup), "--no-cpu-baseline"]
    res = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, timeout=1800)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    if res.returncode != 0 or not lines:
        raise RuntimeError(f"bench.py in {tree} failed ({res.returncode}):\n{res.stdout[-2000:]}\n{res.stderr[-2000:]}")
    out = json.loads(lines[-1])
    return {"frames_per_s": out["value"], "ms_per_step": out.get("ms_per_step")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--bench-rounds", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=200)
    ap.add_argument("--bench-warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    gpu = gpu_info()
    x = torch.from_numpy(np.random.default_rng(0).uniform(-0.5, 0.5, (B, DIMS[0])).astype(np.float32)).to(dev)
    runs = {"off": make_step(False, None, dev), "on": make_step(True, None, dev),
            "clip_off": make_step(False, 1.0, dev), "clip_on": make_step(True, 1.0, dev)}
    for step in runs.values():
        for _ in range(5):
            step(x)
    res = {k: [] for k in runs}
    for _ in range(args.rounds):
        for name, step in runs.items():
            start = step.stats["replays"]
            res[name].append(timed(lambda: step(x), args.steps))
            assert step.stats["replays"] - start == args.steps   # every timed step was a graph replay
    torch.cuda.synchronize()
    for name in ("on", "clip_on"):
        assert int(runs[name].ema.n_averaged) == runs[name].stats["eager"] + runs[name].stats["captures"] + \
            runs[name].stats["replays"]                          # one EMA update per step
    med = {k: float(np.median(v)) for k, v in res.items()}
    out = {"gpu": gpu, "batch": B, "dims": DIMS, "precision": "bf16", "ema_decay": DECAY,
           "steps_per_round": args.steps, "rounds": args.rounds, "step_ms": res, "median_ms": med,
           "ema_cost_ms": {"no_clip": med["on"] - med["off"], "clip": med["clip_on"] - med["clip_off"]},
           "params": runs["off"].model._flat.total,
           "adam_bytes_per_param": {"off": adam_bytes_per_param(False), "on": adam_bytes_per_param(True)}}
    del runs
    torch.cuda.empty_cache()
    if args.parent:
        rows = {"parent": [], "this": []}
        for _ in range(args.bench_rounds):
            rows["parent"].append(bench(args.parent, args))
            rows["this"].append(bench(ROOT, args))
        out["bench"] = {"cmd": f"bench.py --gpus 1 --steps {args.bench_steps} --warmup {args.bench_warmup} "
                               f"--no-cpu-baseline", "rounds": rows,
                        "median_frames_per_s": {k: float(np.median([r["frames_per_s"] for r in v]))
                                                for k, v in rows.items()}}
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_ema_perf.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
