"""Training-step time and launches per step of a model whose dims are padded inside the library, next to the model
it runs as: (S, H, L) = (1024, 2000, 16) runs at (1024, 2048, 64). B = 8192, FusedTrainStep with a CUDA graph.

    python tools/padded_dims_perf.py [--steps 50] [--out DIR]

Prints one JSON object (GPU name and power limit included); --out DIR also writes it to DIR/padded_dims_perf.json."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers are still reported, marked as such
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def measure(dims, batch, steps, warmup):
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import VAE, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = VAE(*dims).to(dev)
    opt = Adam(model.parameters(), lr=1e-4)
    step = FusedTrainStep(model, opt, kl_beta=0.5, graph=True)
    x = (torch.rand(batch, dims[0], device=dev) * 2 - 1) * 0.5
    for _ in range(warmup):
        step(x)
    torch.cuda.synchronize()
    launches = [st["launches"] for st in step._graphs.values()]
    l0 = ops.launch_count(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step(x)
    b.record()
    torch.cuda.synchronize()
    assert step.steady >= steps, "a capture or an eager step fell into the timed window"
    return {"dims": list(dims), "batch": batch, "steps": steps, "step_ms": a.elapsed_time(b) / steps,
            "launches_per_step": launches[0] if len(launches) == 1 else launches,
            "eager_launches_in_window": ops.launch_count(dev) - l0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = dict(gpu_info())
    # alternate the two shapes so that drift of the shared machine affects both alike
    runs = {"padded_1024x2000x16": [], "native_1024x2048x64": []}
    for _ in range(2):
        runs["padded_1024x2000x16"].append(measure((1024, 2000, 16), args.batch, args.steps, args.warmup))
        runs["native_1024x2048x64"].append(measure((1024, 2048, 64), args.batch, args.steps, args.warmup))
    res["runs"] = runs
    res["launches_equal"] = runs["padded_1024x2000x16"][0]["launches_per_step"] == \
        runs["native_1024x2048x64"][0]["launches_per_step"]
    print(json.dumps(res))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "padded_dims_perf.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
