"""Generate tests/golden/* by running the UNMODIFIED reference (imported read-only from /root/reference).

Run in the build container only (`python oracle/gen_golden.py`); the GPU box has no /root/reference, so the
fixtures written here are committed. Test infrastructure - never imported by the product path.

Shims (SURVEY.md 8c): `librosa` is stubbed for the import at rawvae/dataset.py:3 (the dataset classes never call
it); `torchaudio.load` (needs the absent torchcodec) is replaced by a scipy.io.wavfile reader returning
(float32 [C, N] = int16 / 32768, sr); eps is injected by wrapping torch.randn_like (rawvae/model.py:25).
"""
from __future__ import annotations

import hashlib
import importlib.util
import json
import sys
import tempfile
import types
from pathlib import Path

import numpy as np
import torch

REF = Path("/root/reference")
OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"


def load_reference():
    sys.modules.setdefault("librosa", types.ModuleType("librosa"))
    mods = {}
    for name in ("model", "dataset"):
        spec = importlib.util.spec_from_file_location(f"_ref_rawvae_{name}", REF / "rawvae" / f"{name}.py")
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        mods[name] = m
    return mods["model"], mods["dataset"]


class InjectEps:
    """Replace torch.randn_like by a queue of prepared tensors while the reference forward runs."""

    def __init__(self, eps_list):
        self.q = list(eps_list)

    def __enter__(self):
        self.orig = torch.randn_like
        torch.randn_like = lambda t, *a, **k: self.q.pop(0).to(t.dtype)
        return self

    def __exit__(self, *exc):
        torch.randn_like = self.orig


def model_case(ref_model, S, H, L, B, steps, kl_beta, lr, store_full):
    torch.manual_seed(0)
    model = ref_model.VAE(S, H, L)
    gen = torch.Generator().manual_seed(1)
    x = torch.rand(B, S, generator=gen) * 2 - 1
    eps = [torch.randn(B, L, generator=gen) for _ in range(steps)]
    init = {k: v.detach().clone() for k, v in model.state_dict().items()}
    opt = torch.optim.Adam(model.parameters(), lr=lr)
    rec = {}
    losses = []
    for s in range(steps):
        opt.zero_grad()
        with InjectEps([eps[s]]):
            xh, mu, lv = model(x)                                        # train_iterable.py:201
        loss = ref_model.loss_function(xh, x, mu, lv, kl_beta, S)        # train_iterable.py:202
        loss.backward()                                                  # train_iterable.py:208
        if s == 0:
            rec["x_hat"], rec["mu"], rec["logvar"] = xh.detach().clone(), mu.detach().clone(), lv.detach().clone()
            rec["grads"] = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
        losses.append(float(loss))
        opt.step()                                                       # train_iterable.py:210
    final = {k: v.detach().clone() for k, v in model.state_dict().items()}
    ost = opt.state_dict()
    names = [k for k, _ in model.named_parameters()]
    if store_full:
        arrays = {"x": x.numpy(), "eps": torch.stack(eps).numpy(), "losses": np.array(losses, dtype=np.float64),
                  "x_hat": rec["x_hat"].numpy(), "mu": rec["mu"].numpy(), "logvar": rec["logvar"].numpy()}
        for k in names:
            arrays["init/" + k] = init[k].numpy()
            arrays["grad/" + k] = rec["grads"][k].numpy()
            arrays["final/" + k] = final[k].numpy()
            i = names.index(k)
            arrays["exp_avg/" + k] = ost["state"][i]["exp_avg"].numpy()
            arrays["exp_avg_sq/" + k] = ost["state"][i]["exp_avg_sq"].numpy()
        arrays["meta"] = np.array([S, H, L, B, steps], dtype=np.int64)
        arrays["hyper"] = np.array([kl_beta, lr], dtype=np.float64)
        return arrays
    # summary only (default.ini dims are 23 MB of weights - regenerated from the seed at test time)
    def stat(t):
        t = t.double()
        return {"norm": float(t.norm()), "sum": float(t.sum()), "first": [float(v) for v in t.flatten()[:4]]}
    return {"S": S, "H": H, "L": L, "B": B, "steps": steps, "kl_beta": kl_beta, "lr": lr, "losses": losses,
            "n_params": int(sum(p.numel() for p in model.parameters())),
            "x_hat": stat(rec["x_hat"]), "mu": stat(rec["mu"]), "logvar": stat(rec["logvar"]),
            "grads": {k: stat(v) for k, v in rec["grads"].items()},
            "final": {k: stat(v) for k, v in final.items()},
            "state_dict_keys": list(final.keys()),
            "state_dict_shapes": {k: list(v.shape) for k, v in final.items()},
            "optimizer_state_keys": sorted(ost["state"][0].keys()),
            "optimizer_step": float(ost["state"][0]["step"]),
            "param_group": {k: v for k, v in ost["param_groups"][0].items() if k in ("lr", "betas", "eps", "weight_decay", "amsgrad")}}


def digest(a: np.ndarray) -> str:
    """SHA-256 of an array's dtype, shape and bytes."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def small_inputs(S, H, L, B, steps) -> dict:
    """The seeded inputs of model_case: the initial weights of `torch.manual_seed(0); VAE(S, H, L)` (nn.Linear's
    default init in the reference's creation order, rawvae/model.py:13-17), then x and one eps per step drawn from
    Generator seed 1. The caller's global RNG state is left as it was."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        layers = [("fc1", torch.nn.Linear(S, H)), ("fc21", torch.nn.Linear(H, L)), ("fc22", torch.nn.Linear(H, L)),
                  ("fc3", torch.nn.Linear(L, H)), ("fc4", torch.nn.Linear(H, S))]
    out = {f"init/{n}.{w}": getattr(m, w).detach().numpy() for n, m in layers for w in ("weight", "bias")}
    gen = torch.Generator().manual_seed(1)
    out["x"] = (torch.rand(B, S, generator=gen) * 2 - 1).numpy()
    out["eps"] = torch.stack([torch.randn(B, L, generator=gen) for _ in range(steps)]).numpy()
    return out


def split_small(arrays: dict):
    """model_case's arrays as the two files under tests/golden (each under 1 MB): model_small.npz holds the
    reference's outputs and, for the inputs small_inputs regenerates, their digests; model_small_adam.npz holds the
    Adam moments after the last step."""
    regen = [k for k in arrays if k in ("x", "eps") or k.startswith("init/")]
    main = {k: v for k, v in arrays.items() if k not in regen and not k.startswith("exp_avg")}
    main.update({"sha256/" + k: np.array(digest(arrays[k])) for k in regen})
    adam = {k: v for k, v in arrays.items() if k.startswith("exp_avg")}
    return main, adam


def load_small(golden_dir: Path = OUT) -> dict:
    """The arrays model_case returned, from the files split_small wrote. Regenerated inputs are checked against the
    reference's digests; a mismatch (torch's generators no longer reproduce the reference's draws) raises."""
    arrays = dict(np.load(golden_dir / "model_small.npz"))
    arrays.update(np.load(golden_dir / "model_small_adam.npz"))
    S, H, L, B, steps = (int(v) for v in arrays["meta"])
    for k, a in small_inputs(S, H, L, B, steps).items():
        want = str(arrays.pop("sha256/" + k))
        if digest(a) != want:
            raise ValueError(f"regenerated {k} does not reproduce the reference's (sha256 {digest(a)}, want {want})")
        arrays[k] = a
    return arrays


def dataset_case(ref_ds):
    import scipy.io.wavfile as wavfile
    import torchaudio

    rng = np.random.default_rng(1234)
    out = {}
    # map-style datasets on the survey's example length (n = 22 087) and edge lengths
    for n in (22087, 1024, 1025, 2048, 1151, 1152):
        audio = (rng.standard_normal(n) * 0.1).astype(np.float32)
        ds = ref_ds.AudioDataset(audio, 1024, 44100, 128, transform=ref_ds.ToTensor())
        ts = ref_ds.TestDataset(audio, 1024, 44100, transform=ref_ds.ToTensor())
        out[f"audio_{n}"] = audio
        out[f"audio_len_{n}"] = np.array([len(ds), len(ts)], dtype=np.int64)
        idx = sorted({0, len(ds) - 1, len(ds) // 2, min(7, len(ds) - 1)})
        out[f"audio_idx_{n}"] = np.array(idx, dtype=np.int64)
        out[f"audio_frames_{n}"] = np.stack([ds[i].numpy() for i in idx])
        out[f"test_frames_{n}"] = np.stack([ts[i].numpy() for i in range(len(ts))])
    # segment_length not a multiple of hop -> ValueError (dataset.py:99-100)
    try:
        ref_ds.AudioDataset(np.zeros(4096, dtype=np.float32), 1000, 44100, 128)
        out["raises_valueerror"] = np.array([0])
    except ValueError:
        out["raises_valueerror"] = np.array([1])

    # streaming dataset: three PCM16 wavs (one stereo, one at 22.05 kHz -> resampled) in sorted glob order
    def fake_load(path):
        sr, data = wavfile.read(str(path))
        data = data.astype(np.float32) / 32768.0
        data = data[None, :] if data.ndim == 1 else data.T
        return torch.from_numpy(np.ascontiguousarray(data)), sr

    orig_load = torchaudio.load
    torchaudio.load = fake_load
    try:
        with tempfile.TemporaryDirectory() as td:
            td = Path(td)
            lens = {"a.wav": 3000, "b.wav": 5000, "c.wav": 2200}
            pcm = {}
            for name, n in lens.items():
                v = np.clip(np.round(rng.standard_normal(n) * 3000), -32768, 32767).astype(np.int16)
                if name == "b.wav":
                    v = np.stack([v, -v], axis=1)  # stereo: channel 0 kept (dataset.py:54-55)
                wavfile.write(str(td / name), 44100, v)
                pcm[name] = v
            ds = ref_ds.IterableAudioDataset(td, 44100, 128, torch.float32, torch.device("cpu"), shuffle=False)
            order = [p.name for p in ds.audio_file_list]
            it = iter(ds)
            frames = torch.stack([next(it) for _ in range(150)]).numpy()  # > one cycle (17 + 33 + 10 = 60 frames)
            out["stream_order"] = np.array(order)
            out["stream_frames"] = frames
            for name in lens:
                out["stream_pcm_" + name] = pcm[name]
    finally:
        torchaudio.load = orig_load
    return out


def main():
    OUT.mkdir(parents=True, exist_ok=True)
    ref_model, ref_ds = load_reference()
    small, adam = split_small(model_case(ref_model, S=128, H=192, L=64, B=48, steps=3, kl_beta=1e-4, lr=1e-3,
                                         store_full=True))
    np.savez_compressed(OUT / "model_small.npz", **small)
    np.savez_compressed(OUT / "model_small_adam.npz", **adam)
    # default.ini dims (default.ini:5,18-20,26): summary statistics only
    default = model_case(ref_model, S=1024, H=2048, L=256, B=256, steps=2, kl_beta=1e-4, lr=1e-4, store_full=False)
    (OUT / "model_default_summary.json").write_text(json.dumps(default, indent=1))
    np.savez_compressed(OUT / "dataset.npz", **dataset_case(ref_ds))
    print("wrote", sorted(p.name for p in OUT.iterdir()))


if __name__ == "__main__":
    main()
