"""Cost of gradient-norm clipping in the fused training step: steady-state CUDA-graph steps of FusedTrainStep at
B = 8192 and the default dims (1024, 2048, 256), bf16, without clipping, with a binding max_grad_norm, and with
max_grad_norm = inf (measure only). The three runs alternate within one process, `--rounds` times, each timing
`--steps` replayed steps with CUDA events after a warm-up that captures the graph. Also the norm reduction alone
(rvae_plan_grad_norm over the flat gradient buffer, 4 B/param read) in bytes/s, over `--norm-reps` back-to-back
calls; the 23 MB buffer fits the 126 MB L2, so that rate is L2-warm, as the reduction runs inside a step.

    python tools/clip_perf.py [--steps 200] [--rounds 3] [--norm-reps 2000] [--out DIR]

Prints one JSON object (GPU name and power limit included); --out DIR also writes it to DIR/r3_clip_perf.json."""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from padded_dims_perf import gpu_info  # noqa: E402

B, DIMS = 8192, (1024, 2048, 256)
BINDING = 5e-5   # below the gradient norm of every timed step (2e-4 to 7e-4 around step 300 on a B200): it binds


def make_step(max_grad_norm, dev):
    from rawaudiovae_kelsey_b200.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    torch.manual_seed(0)
    model = VAE(*DIMS, precision="bf16").to(dev)
    model.eps_seed = 1
    opt = Adam(model.parameters(), lr=1e-4)
    return FusedTrainStep(model, opt, kl_beta=1e-4, graph=True, max_grad_norm=max_grad_norm)


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--norm-reps", type=int, default=2000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    x = torch.from_numpy(np.random.default_rng(0).uniform(-0.5, 0.5, (B, DIMS[0])).astype(np.float32)).to(dev)
    runs = {"off": make_step(None, dev), "binding": make_step(BINDING, dev), "inf": make_step(math.inf, dev)}
    for step in runs.values():
        for _ in range(5):
            step(x)
    res = {k: [] for k in runs}
    for _ in range(args.rounds):
        for name, step in runs.items():
            start = step.stats["replays"]
            res[name].append(timed(lambda: step(x), args.steps))
            assert step.stats["replays"] - start == args.steps   # every timed step was a graph replay
    norms = {k: float(s.grad_norm) for k, s in runs.items() if s.grad_norm is not None}
    assert norms["binding"] > BINDING, norms   # the "binding" run did clip
    # the reduction alone, on the gradient of a real step (keep_grads: the buffer is not cleared)
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    model, opt = runs["off"].model, runs["off"].optimizer
    FusedTrainStep(model, opt, kl_beta=1e-4, keep_grads=True)(x)
    plan = model._load(x)
    out_t = torch.empty((), dtype=torch.float32, device=dev)
    for _ in range(20):
        plan.grad_norm(out_t)
    norm_ms = timed(lambda: plan.grad_norm(out_t), args.norm_reps)
    flat = model._flat
    nbytes = 4 * flat.total
    out = {"gpu": gpu_info(), "batch": B, "dims": DIMS, "precision": "bf16", "steps_per_round": args.steps,
           "binding_max_grad_norm": BINDING, "last_grad_norm": norms,
           "step_ms": res, "median_ms": {k: float(np.median(v)) for k, v in res.items()},
           "norm_reduction": {"params": flat.total, "bytes": nbytes, "ms": norm_ms,
                              "bytes_per_s": nbytes / (norm_ms * 1e-3), "reps": args.norm_reps,
                              "note": "four launches (W4 | W3 | W2 + biases | W1) and the "
                                      "finalisation, as in a step; L2-warm: the 23 MB buffer fits the 126 MB L2"}}
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_clip_perf.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
