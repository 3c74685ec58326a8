"""Pin the CPU oracle (oracle/rawvae_oracle.py) against outputs of the reference itself (tests/golden/*,
written by oracle/gen_golden.py from the unmodified reference code). CPU only."""
import json

import numpy as np
import pytest
import torch

from oracle import gen_golden
from oracle import rawvae_oracle as O


def _rel(a, b):
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


@pytest.fixture(scope="module")
def small(golden_dir):
    return gen_golden.load_small(golden_dir)


def _params(small, prefix, dtype):
    return {k: torch.from_numpy(small[f"{prefix}/{k}"]).to(dtype) for k in O.PARAM_NAMES}


def test_init_matches_reference_default_init(small):
    S, H, L, B, steps = small["meta"]
    p = O.init_params(int(S), int(H), int(L), seed=0)
    for k in O.PARAM_NAMES:
        np.testing.assert_array_equal(p[k].numpy(), small["init/" + k])


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 2e-6), (torch.float32, 2e-6)])
def test_forward_loss_backward(small, dtype, tol):
    S, H, L, B, steps = (int(v) for v in small["meta"])
    kl_beta, lr = (float(v) for v in small["hyper"])
    p = _params(small, "init", dtype)
    x = torch.from_numpy(small["x"]).to(dtype)
    eps = torch.from_numpy(small["eps"][0]).to(dtype)
    act = O.forward(p, x, eps)
    assert _rel(act["x_hat"], small["x_hat"]) < tol
    assert _rel(act["mu"], small["mu"]) < tol
    assert _rel(act["logvar"], small["logvar"]) < tol
    loss = O.loss_function(act["x_hat"], x, act["mu"], act["logvar"], kl_beta, S)
    assert abs(float(loss) - float(small["losses"][0])) < 1e-6 * abs(float(small["losses"][0]))
    g = O.backward(p, act, kl_beta)
    for k in O.PARAM_NAMES:
        assert _rel(g[k], small["grad/" + k]) < 5e-6, k


def test_adam_three_steps(small):
    S, H, L, B, steps = (int(v) for v in small["meta"])
    kl_beta, lr = (float(v) for v in small["hyper"])
    p = _params(small, "init", torch.float64)
    st = O.adam_init(p)
    x = torch.from_numpy(small["x"]).double()
    for s in range(steps):
        loss = O.train_step(p, st, x, torch.from_numpy(small["eps"][s]).double(), kl_beta, lr)
        assert abs(loss - float(small["losses"][s])) < 2e-6 * abs(float(small["losses"][s]))
    for k in O.PARAM_NAMES:
        assert _rel(p[k], small["final/" + k]) < 1e-6, k
        assert _rel(st[k]["exp_avg"], small["exp_avg/" + k]) < 1e-5, k
        assert _rel(st[k]["exp_avg_sq"], small["exp_avg_sq/" + k]) < 1e-5, k


def test_default_ini_dims_summary(golden_dir):
    """default.ini dimensions (1024/2048/256): weights regenerated from the seed, compared through statistics."""
    g = json.loads((golden_dir / "model_default_summary.json").read_text())
    S, H, L, B = g["S"], g["H"], g["L"], g["B"]
    assert g["n_params"] == 5772800  # SURVEY.md 8a (a1)
    assert g["state_dict_keys"] == list(O.PARAM_NAMES)
    assert g["state_dict_shapes"]["fc21.weight"] == [L, H] and g["state_dict_shapes"]["fc4.weight"] == [S, H]
    p = O.init_params(S, H, L, seed=0)
    gen = torch.Generator().manual_seed(1)
    x = torch.rand(B, S, generator=gen) * 2 - 1
    eps = [torch.randn(B, L, generator=gen) for _ in range(g["steps"])]
    st = O.adam_init(p)
    act = O.forward(p, x, eps[0])
    for name in ("x_hat", "mu", "logvar"):
        assert abs(float(act[name].double().norm()) - g[name]["norm"]) < 2e-5 * g[name]["norm"]
    gr = O.backward(p, act, g["kl_beta"])
    for k in O.PARAM_NAMES:
        assert abs(float(gr[k].double().norm()) - g["grads"][k]["norm"]) < 1e-4 * g["grads"][k]["norm"], k
    for s in range(g["steps"]):
        loss = O.train_step(p, st, x, eps[s], g["kl_beta"], g["lr"])
        assert abs(loss - g["losses"][s]) < 1e-5 * abs(g["losses"][s])
    for k in O.PARAM_NAMES:
        assert abs(float(p[k].double().norm()) - g["final"][k]["norm"]) < 1e-5 * g["final"][k]["norm"], k
    assert g["optimizer_state_keys"] == ["exp_avg", "exp_avg_sq", "step"] and g["optimizer_step"] == g["steps"]
    assert g["param_group"]["betas"] == [0.9, 0.999] and g["param_group"]["eps"] == 1e-8


# ------------------------------------------------------------------------------------------------ framing
@pytest.fixture(scope="module")
def ds(golden_dir):
    return np.load(golden_dir / "dataset.npz")


@pytest.mark.parametrize("n", [22087, 1024, 1025, 2048, 1151, 1152])
def test_map_style_framing_bit_exact(ds, n):
    audio = ds[f"audio_{n}"]
    n_audio, n_test = (int(v) for v in ds[f"audio_len_{n}"])
    assert O.audio_dataset_len(n, 1024, 128) == n_audio
    idx = [int(i) for i in ds[f"audio_idx_{n}"]]
    np.testing.assert_array_equal(O.audio_dataset_frames(audio, 1024, 128, idx), ds[f"audio_frames_{n}"])
    tf = O.test_dataset_frames(audio, 1024)
    assert len(tf) == n_test
    np.testing.assert_array_equal(tf, ds[f"test_frames_{n}"])


def test_known_answers_from_survey():
    assert O.audio_dataset_len(22087, 1024, 128) == 166       # SURVEY.md Appendix B
    assert len(O.test_dataset_frames(np.zeros(22087, np.float32), 1024)) == 22
    assert len(O.iterable_file_frames(np.zeros(3000, np.float32), 128)) == 17
    assert len(O.iterable_file_frames(np.zeros(5000, np.float32), 128)) == 33


def test_hop_must_divide_segment(ds):
    assert int(ds["raises_valueerror"][0]) == 1
    with pytest.raises(ValueError):
        O.audio_dataset_len(4096, 1000, 128)


def test_stream_order_and_frames_bit_exact(ds):
    order = [str(s) for s in ds["stream_order"]]
    files = []
    for name in order:
        pcm = ds["stream_pcm_" + name]
        mono = pcm[:, 0] if pcm.ndim == 2 else pcm            # channel 0 (dataset.py:54-55)
        files.append(mono.astype(np.float32) / 32768.0)
    got = O.iterable_stream(files, 128, 150)
    np.testing.assert_array_equal(got, ds["stream_frames"])


def test_resynthesis_identities(ds):
    audio = ds["audio_22087"]
    tf = O.test_dataset_frames(audio, 1024)
    np.testing.assert_array_equal(O.resynth_concat(tf), O.pad_to_multiple(audio, 1024))
    fr = O.audio_dataset_frames(audio, 1024, 128)
    ola = O.resynth_overlap_add(fr, 128)
    np.testing.assert_allclose(ola, O.pad_to_multiple(audio, 128).astype(np.float64), rtol=0, atol=1e-7)
    # hop == S degenerates to concatenation
    np.testing.assert_allclose(O.resynth_overlap_add(tf, 1024), O.resynth_concat(tf).astype(np.float64))
