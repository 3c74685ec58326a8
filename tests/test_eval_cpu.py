"""Held-out evaluation without a GPU: the rvae_frame_loss entry point rejects malformed arguments before it needs a
device, and the trainers' [training] test_loss key."""
import configparser

import pytest

from rawaudiovae_kelsey_b200 import _lib

GOOD = dict(ctx=None, xhat=256, ld_xhat=1024, mu=512, logvar=768, ld_lat=64, rows=10, S=1024, L=64, audio=1024,
            audio_is_i16=0, n_samples=5000, first_frame=0, hop=128, rec=2048, kl=4096)


def _call(**over):
    a = dict(GOOD, **over)
    lib = _lib.load()
    rc = lib.rvae_frame_loss(a["ctx"], a["xhat"], a["ld_xhat"], a["mu"], a["logvar"], a["ld_lat"], a["rows"], a["S"],
                             a["L"], a["audio"], a["audio_is_i16"], a["n_samples"], a["first_frame"], a["hop"],
                             a["rec"], a["kl"], None)
    return rc, lib.rvae_last_error().decode()


def test_frame_loss_is_exported_with_a_signature():
    lib = _lib.load()
    assert hasattr(lib, "rvae_frame_loss") and "rvae_frame_loss" in _lib.SIGNATURES
    assert lib.rvae_abi_version() == 5


@pytest.mark.parametrize("over, words", [
    ({"xhat": None}, "null"), ({"mu": None}, "null"), ({"logvar": None}, "null"), ({"audio": None}, "null"),
    ({"rec": None}, "null"), ({"kl": None}, "null"),
    ({"rows": 0}, "rows"), ({"rows": -3}, "rows"), ({"S": 0}, "S 0"), ({"L": -1}, "L -1"),
    ({"ld_xhat": 1000}, "ld_xhat"), ({"ld_lat": 63}, "ld_lat"),
    ({"hop": 0}, "hop"), ({"n_samples": -1}, "n_samples"), ({"first_frame": -2}, "first_frame"),
])
def test_frame_loss_rejects_malformed_arguments(over, words):
    rc, msg = _call(**over)
    assert rc == 1, msg
    assert "frame_loss" in msg and words in msg, msg


def test_frame_loss_with_valid_arguments_needs_a_context():
    rc, msg = _call()
    assert rc == 1 and "rvae_ctx" in msg


def _config(test_loss=None, generate_test=True):
    c = configparser.ConfigParser(allow_no_value=True)
    c.read_string("[dataset]\ngenerate_test = {}\n[training]\nbatch_size = 4\n".format(generate_test))
    if test_loss is not None:
        c["training"]["test_loss"] = str(test_loss)
    return c


def test_test_loss_key_defaults_to_false():
    from rawaudiovae_kelsey_b200.trainer import _test_loss_enabled
    assert _test_loss_enabled(_config()) is False
    assert _test_loss_enabled(_config(generate_test=False)) is False
    assert _test_loss_enabled(_config(False)) is False
    assert _test_loss_enabled(_config(True)) is True


@pytest.mark.parametrize("which", ["epoch", "stream"])
def test_test_loss_without_generate_test_raises_at_start_up(tmp_path, which):
    from rawaudiovae_kelsey_b200 import trainer
    with pytest.raises(ValueError, match="generate_test"):
        trainer._test_loss_enabled(_config(True, generate_test=False))
    (tmp_path / "data" / "test_audio").mkdir(parents=True)
    ini = tmp_path / "t.ini"
    ini.write_text(f"""[audio]
sampling_rate = 44100
hop_length = 128
segment_length = 1024
[dataset]
datapath = {tmp_path / 'data'}
test_dataset = test_audio
generate_test = False
run_number = 0
[VAE]
latent_dim = 64
n_units = 256
kl_beta = 0.0001
[training]
epochs = 1
total_num_frames = 1024
save_best_model_after = 0
learning_rate = 0.0001
batch_size = 256
checkpoint_interval = 1
test_loss = True
[extra]
description = t
""")
    run = trainer.run_epoch_trainer if which == "epoch" else trainer.run_stream_trainer
    with pytest.raises(ValueError, match="generate_test"):   # before any device or dataset work
        run(["--config", str(ini)])
    assert not (tmp_path / "data" / "t").exists()
