"""Cost of deterministic training steps: steady-state CUDA-graph steps of FusedTrainStep at the default dims
(1024, 2048, 256) with deterministic off and on, alternated within one process `--rounds` times, each timing `--steps`
replayed steps with CUDA events after a warm-up that captures the graph. Three workloads: B = 8192 gathered frames in
bf16 and in fp32 mode, and B = 4096 consecutive frames read in place (bf16). The next batch is prefetched by every
step, as the trainers and bench.py run. Also the scratch bytes of the deterministic plan.

    python tools/deterministic_perf.py [--steps 200] [--rounds 3] [--profile-steps 20] [--out DIR]

After the timed rounds, `--profile-steps` more replayed steps of each mode run under torch.profiler (CUDA activities,
a pass of its own, not timed): the GPU time per step of every kernel name, so the cost of the mode can be attributed.

Prints one JSON object (GPU name and power limit included); --out DIR also writes it to
DIR/r3_deterministic_perf.json."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from padded_dims_perf import gpu_info  # noqa: E402

DIMS, HOP = (1024, 2048, 256), 128
WORKLOADS = {"bf16_gather_8192": ("bf16", 8192, False), "fp32_gather_8192": ("fp32", 8192, False),
             "bf16_in_place_4096": ("bf16", 4096, True)}


class Run:
    """One step object fed a fixed cycle of batches, each step prefetching the next."""

    def __init__(self, precision, batch, in_place, deterministic, audio, dev):
        from rawaudiovae_kelsey_b200.model import VAE, FrameBatch, FusedTrainStep
        from rawaudiovae_kelsey_b200.optim import Adam
        torch.manual_seed(0)
        model = VAE(*DIMS, precision=precision).to(dev)
        model.eps_seed = 1
        self.step = FusedTrainStep(model, Adam(model.parameters(), lr=1e-4), kl_beta=1e-4, graph=True,
                                   deterministic=deterministic)
        n = audio.numel() // HOP - DIMS[0] // HOP
        gen = torch.Generator().manual_seed(1)
        if in_place:
            self.batches = [FrameBatch(audio, batch, HOP, DIMS[0], first_frame=(i * 7919) % (n - batch)) for i in range(2)]
        else:
            self.batches = [FrameBatch(audio, batch, HOP, DIMS[0],
                                       frame_idx=torch.randint(0, n, (batch,), generator=gen).to(dev)) for _ in range(2)]
        self.i = 0

    def __call__(self):
        cur, nxt = self.batches[self.i % 2], self.batches[(self.i + 1) % 2]
        self.step(cur, next_data=nxt)
        self.i += 1


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def kernel_profile(run, steps):
    """GPU time per step (us) of each kernel name over `steps` replayed steps, largest first."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            run()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "self_device_time_total", None)
        if t is None:
            t = ev.self_cuda_time_total
        if t > 0:
            out[ev.key[:120]] = out.get(ev.key[:120], 0.0) + t / steps
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile-steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    audio = torch.from_numpy(np.random.default_rng(0).uniform(-0.5, 0.5, 3 * 8192 * HOP).astype(np.float32)).to(dev)
    out = {"gpu": gpu_info(), "dims": DIMS, "steps_per_round": args.steps, "rounds": args.rounds, "workloads": {}}
    for name, (precision, batch, in_place) in WORKLOADS.items():
        runs = {mode: Run(precision, batch, in_place, mode == "on", audio, dev) for mode in ("off", "on")}
        for r in runs.values():
            for _ in range(6):
                r()
        res = {k: [] for k in runs}
        for _ in range(args.rounds):
            for mode, r in runs.items():
                start = r.step.stats["replays"]
                res[mode].append(timed(r, args.steps))
                assert r.step.stats["replays"] - start == args.steps   # every timed step was a graph replay
        prof = {mode: kernel_profile(r, args.profile_steps) for mode, r in runs.items()} if args.profile_steps else {}
        plan = runs["on"].step.model._plan_for(batch)
        med = {k: float(np.median(v)) for k, v in res.items()}
        out["workloads"][name] = {"precision": precision, "batch": batch, "in_place": in_place, "step_ms": res,
                                  "median_ms": med, "cost": med["on"] / med["off"] - 1.0,
                                  "scratch_bytes": plan.deterministic_bytes(), "plan_max_batch": plan.max_batch,
                                  "kernel_us_per_step": prof}
        del runs
        torch.cuda.empty_cache()
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_deterministic_perf.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
