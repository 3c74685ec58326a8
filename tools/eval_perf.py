"""Cost of held-out evaluation: inference.evaluate_audio next to inference.reconstruct_audio on the same audio
(AudioDataset framing at hop 128, 262 144 frames, batch 16384, float32 audio) at the default dims (1024, 2048, 256)
and the widened config (4096, 4096, 256), and the per-frame loss kernel (rvae_frame_loss) alone with its achieved
bandwidth over the bytes it must move: 4 S (xhat) + 8 L (mu, logvar) + 4 hop (the audio each frame adds) + 8 (two
results) per frame. The kernel's inputs are > 256 MB, so they come from HBM, not the 126 MB L2.

    python tools/eval_perf.py [--repeats 3] [--out DIR]

Prints one JSON object (GPU name and power limit included); --out DIR also writes it to DIR/eval_perf.json."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from padded_dims_perf import gpu_info  # noqa: E402

HOP, FRAMES, BATCH = 128, 262144, 16384


def timed(fn, repeats):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def measure(dims, repeats):
    from rawaudiovae_kelsey_b200 import inference as I
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import VAE
    dev = torch.device("cuda", 0)
    S, H, L = dims
    torch.manual_seed(0)
    model = VAE(S, H, L).to(dev)
    g = torch.Generator(device=dev).manual_seed(1)
    wav = (torch.rand((FRAMES - 1) * HOP + S, generator=g, device=dev) * 2 - 1) * 0.5
    assert I.frame_count(wav.numel(), S, HOP) == FRAMES
    ev = lambda: I.evaluate_audio(model, wav, 1e-4, hop=HOP, batch_size=BATCH)
    rc = lambda: I.reconstruct_audio(model, wav, hop=HOP, batch_size=BATCH)
    ev()
    rc()   # warm-up: plans, tensor maps, module loads
    t_ev, t_rc = [], []
    for _ in range(repeats):   # alternate the two so that drift of the shared machine affects both alike
        t_ev += timed(ev, 1)
        t_rc += timed(rc, 1)
    # the kernel alone, on inputs larger than L2, cycling through first_frame offsets
    rows = max(BATCH, (1 << 28) // (4 * S))
    xh = torch.rand(rows, S, device=dev, generator=g)
    mu = torch.randn(rows, L, device=dev, generator=g)
    lv = torch.randn(rows, L, device=dev, generator=g)
    audio = torch.rand((rows * 2) * HOP + S, device=dev, generator=g)
    rec = torch.empty(rows, device=dev)
    kl = torch.empty(rows, device=dev)
    launches = 20
    k = lambda: [ops.frame_loss(xh, mu, lv, audio, (i % 2) * rows, HOP, rec, kl) for i in range(launches)]
    k()
    t_k = [t / launches for t in timed(k, repeats)]
    nbytes = rows * (4 * S + 8 * L + 4 * HOP + 8)
    best = min(t_k)
    return {"dims": list(dims), "frames": FRAMES, "hop": HOP, "batch": BATCH,
            "evaluate_audio_ms": t_ev, "reconstruct_audio_ms": t_rc,
            "evaluate_over_reconstruct": min(t_ev) / min(t_rc),
            "frame_loss_kernel": {"rows": rows, "ms": t_k, "algorithmic_bytes": nbytes,
                                  "GB_per_s": nbytes / (best * 1e-3) / 1e9}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = dict(gpu_info())
    res["runs"] = [measure(d, args.repeats) for d in ((1024, 2048, 256), (4096, 4096, 256))]
    print(json.dumps(res))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "eval_perf.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
