"""The two training drivers of the reference, `train.py` (epochs over a map-style AudioDataset) and
`train_iterable.py` (a fixed number of batches over the streaming IterableAudioDataset), with the same CLI
(`--config x.ini`), ini schema (default.ini / kelsey_iterable.ini) and on-disk artefacts:

    <datapath>/<description>/run-NNN/{config.ini, console_log, logs/, audio_logs/{<test>.txt, test_original.wav,
        test_reconst_NNNNN.wav}, model/checkpoints/ckpt_NNNNN, model/best_model.pt, model/last_model.pt}

(reference: train.py:32-307, train_iterable.py:34-329). What changed underneath: the wav corpus lives in HBM, batches
are FrameBatch descriptors framed on the GPU, one FusedTrainStep call replaces zero_grad/forward/loss/backward/step,
and losses are read back in blocks instead of three `.item()` syncs per batch. Reference bugs that prevented the
scripts from running at all are fixed forward (SURVEY.md Q1-Q4): the model really goes to the GPU, the checkpoint
branch no longer raises NameError / TypeError, `generate_test` is parsed as a boolean. Under torchrun
(WORLD_SIZE > 1) the same scripts train data-parallel; rank 0 writes the artefacts.
"""
from __future__ import annotations

import argparse
import configparser
import os
import random
import sys
import time
from itertools import islice
from pathlib import Path

import numpy as np
import torch

from . import audio_io, dist as rdist
from .dataset import AudioDataset, IterableAudioDataset, ToTensor
from .inference import evaluate_audio
from .ema import ExponentialMovingAverage, check_ema_decay
from .model import VAE, FusedTrainStep, check_max_grad_norm
from .optim import Adam
from .schedule import Schedule
from .stats import ParamHistogramLogger
from .testaudio import init_test_audio


class Tee:
    """stdout -> console + <workdir>/console_log (train_iterable.py:117-133)."""

    def __init__(self, *files):
        self.files = files

    def write(self, obj):
        for f in self.files:
            f.write(obj)
            f.flush()

    def flush(self):
        for f in self.files:
            f.flush()


class _NullWriter:
    def __getattr__(self, name):
        return lambda *a, **k: None


def _summary_writer(log_dir, enabled: bool):
    if not enabled:
        return _NullWriter()
    try:
        from torch.utils.tensorboard import SummaryWriter
        return SummaryWriter(log_dir=log_dir)
    except Exception as e:  # tensorboard not installed: keep training, say so once
        print("TensorBoard unavailable ({}); scalar logging disabled".format(e))
        return _NullWriter()


def _read_config(argv):
    parser = argparse.ArgumentParser()
    parser.add_argument('--config', type=str, default='./default.ini', help='path to the config file')
    args = parser.parse_args(argv)
    config = configparser.ConfigParser(allow_no_value=True)
    if not config.read(args.config):
        print('Config File Not Found at {}'.format(args.config))
        sys.exit(1)
    return config


def _make_workspace(config, dataset: Path, rank: int):
    """First free <datapath>/<description>/run-NNN with NNN >= run_number (train.py:94-111)."""
    desc = config['extra'].get('description')
    run_id = config['dataset'].getint('run_number')
    if rank != 0:
        return None
    while True:
        workdir = dataset / desc / 'run-{:03d}'.format(run_id)
        try:
            os.makedirs(workdir)
            break
        except OSError:
            if workdir.is_dir():
                run_id += 1
                continue
            raise
    config['dataset']['workspace'] = str(workdir.resolve())
    print("Workspace: {}".format(workdir))
    return workdir


def _common_setup(config):
    rank, world, local_rank = rdist.init_from_env()
    if not torch.cuda.is_available():
        raise RuntimeError("rawaudiovae_kelsey_b200 trains on a CUDA device (sm_100a); there is no CPU fallback")
    device = torch.device('cuda', local_rank)
    torch.cuda.set_device(device)
    device_name = torch.cuda.get_device_name(device)
    print('Device: {}'.format(device_name))
    config['VAE']['device_name'] = device_name
    return rank, world, device


def _reconstruct_test(model, test_dataset, batch_size, device):
    """model(test_sample)[0] over the TestDataset, concatenated and flattened (train_iterable.py:228-246)."""
    preds = []
    with torch.no_grad():
        for fb in test_dataset.gpu_loader(batch_size, device):
            preds.append(model(fb)[0])
    return torch.cat(preds, 0).view(-1).cpu().numpy()


def _precision(config) -> str:
    return config['VAE'].get('precision', fallback='bf16')


def _test_loss_enabled(config) -> bool:
    """[training] test_loss (optional, default False): score the held-out set at every checkpoint, log it and choose
    best_model.pt by it. The held-out audio is only loaded when [dataset] generate_test is on."""
    on = config['training'].getboolean('test_loss', fallback=False)
    if on and not config['dataset'].getboolean('generate_test'):
        raise ValueError("[training] test_loss = True needs [dataset] generate_test = True: the test set is only "
                         "loaded for it")
    return on


def _schedule(config, total_steps: int) -> Schedule:
    """The run's learning-rate and KL-weight schedule over total_steps steps: [training] lr_schedule, lr_warmup_steps,
    lr_min and [VAE] kl_anneal, kl_beta_start, kl_anneal_steps (default: the whole run), kl_cycles, kl_cycle_ratio.
    Missing keys give the constant schedule of the reference; bad values raise ValueError."""
    tr, vae = config['training'], config['VAE']
    return Schedule(lr_schedule=tr.get('lr_schedule', fallback='constant'),
                    warmup_steps=tr.getint('lr_warmup_steps', fallback=0),
                    total_steps=total_steps,
                    lr_min=tr.getfloat('lr_min', fallback=0.0),
                    kl_anneal=vae.get('kl_anneal', fallback='constant'),
                    kl_beta_start=vae.getfloat('kl_beta_start', fallback=0.0),
                    kl_anneal_steps=vae.getint('kl_anneal_steps', fallback=max(total_steps, 1)),
                    kl_cycles=vae.getint('kl_cycles', fallback=1),
                    kl_cycle_ratio=vae.getfloat('kl_cycle_ratio', fallback=0.5))


def _max_grad_norm(config):
    """[training] max_grad_norm (optional): clip each step's gradient by its global L2 norm at this value, and log the
    pre-clip norm as 'Grad Norm'; inf logs without clipping. Absent or empty: no clipping, no extra tag. Values <= 0,
    NaN or text that is not a number raise ValueError."""
    v = config['training'].get('max_grad_norm', fallback='').strip()
    if not v:
        return None
    try:
        f = float(v)
    except ValueError:
        raise ValueError(f"[training] max_grad_norm must be a number > 0 or inf, got {v!r}") from None
    return check_max_grad_norm(f)


def _ema_decay(config):
    """[training] ema_decay (optional): keep an exponential moving average of the weights with this decay, in [0, 1]
    (ema.ExponentialMovingAverage, updated inside every training step). The test reconstructions, the test loss,
    best_model.pt and last_model.pt then use the averaged weights, and each checkpoint also holds them
    ('ema_state_dict', 'ema_n_averaged'). Absent or empty: no average. Values outside [0, 1], NaN or text that is not a
    number raise ValueError."""
    v = config['training'].get('ema_decay', fallback='').strip()
    if not v:
        return None
    try:
        f = float(v)
    except ValueError:
        raise ValueError(f"[training] ema_decay must be a number in [0, 1], got {v!r}") from None
    try:
        return check_ema_decay(f)
    except ValueError:
        raise ValueError(f"[training] ema_decay must be in [0, 1], got {v!r}") from None


def _with_ema(state, ema):
    """A checkpoint dict, plus the average's weights and update count when an EMA is kept."""
    if ema is not None:
        state['ema_state_dict'] = ema.state_dict()
        state['ema_n_averaged'] = int(ema.n_averaged.item())
    return state


def _deterministic(config) -> bool:
    """[training] deterministic (optional bool, default False): bitwise reproducible training steps (FusedTrainStep /
    DataParallelTrainStep deterministic=True). A value that is not a boolean raises ValueError."""
    v = config['training'].get('deterministic', fallback='').strip()
    if not v:
        return False
    try:
        return config['training'].getboolean('deterministic')
    except ValueError:
        raise ValueError(f"[training] deterministic must be a boolean (True / False), got {v!r}") from None


def _seed(config):
    """[training] seed (optional int): seeds torch and random at start-up, which fixes the initial weights, the
    sampler permutation, the stream's file order and the noise seed. Absent or empty: unseeded. Text that is not an
    integer raises ValueError."""
    v = config['training'].get('seed', fallback='').strip()
    if not v:
        return None
    try:
        return int(v)
    except ValueError:
        raise ValueError(f"[training] seed must be an integer, got {v!r}") from None


def _apply_seed(seed) -> None:
    if seed is not None:
        torch.manual_seed(seed)
        random.seed(seed)


def _epoch_steps(n_frames: int, batch_size: int, world: int = 1) -> int:
    """Training steps per epoch of GpuFrameLoader (drop_last=False): a last global batch with fewer frames than ranks
    is skipped."""
    n = -(-n_frames // batch_size)
    return n - 1 if n > 0 and n_frames - (n - 1) * batch_size < world else n


def _epoch_trainer_steps(config, n_frames: int, world: int = 1) -> int:
    """Steps of a run_epoch_trainer run over a training set of n_frames frames: epochs x steps per epoch."""
    return config['training'].getint('epochs') * _epoch_steps(n_frames, config['training'].getint('batch_size'), world)


def _stream_trainer_steps(config) -> int:
    """Steps of a run_stream_trainer run: total_num_batches (train_iterable.py:74)."""
    return int(config['training'].getint('total_num_frames') / config['training'].getint('batch_size'))


def _log_hparams(writer, schedule, optimizer, kl_beta, batch_id):
    """The learning rate the step at batch_id applies and, when it is annealed, its KL weight."""
    writer.add_scalar('Learning Rate', schedule.lr_at(batch_id, optimizer.param_groups[0]['lr']), batch_id)
    if schedule.kl_anneal != 'constant':
        writer.add_scalar('KL Beta', schedule.beta_at(batch_id, kl_beta), batch_id)


def _evaluate_test(model, test_dataset, kl_beta, batch_size, writer, step_id):
    """Held-out loss of the current weights (inference.evaluate_audio over the TestDataset, Philox seed 0, so every
    checkpoint sees the same noise), logged under Loss/test*. batch_size = the training batch: the training plan is
    reused, no new workspace."""
    ev = evaluate_audio(model, test_dataset.audio_np, kl_beta, batch_size=batch_size, seed=0)
    writer.add_scalar('Loss/test', ev.loss, step_id)
    writer.add_scalar('Loss/test_reconstruction', ev.reconstruction_mean, step_id)
    writer.add_scalar('Loss/test_kl', ev.kl_mean, step_id)
    print('Test loss: {:.9f} - reconstruction: {:.9f} - KL: {:.9f}'.format(ev.loss, ev.reconstruction_mean,
                                                                            ev.kl_mean))
    return ev.loss


def _keep_best_test(model, t_loss, best, workdir, config, key, step_id):
    """best_model.pt by held-out loss: saves the model and records config[training][key] = step_id and best_test_loss
    when t_loss beats `best`. Returns the best test loss so far."""
    if t_loss >= best:
        return best
    save_path = workdir.joinpath('model').joinpath('best_model.pt')
    torch.save(model, save_path)
    print('{} {:05d}: Saved {} (test loss {:.9f})'.format(key, step_id, save_path, t_loss))
    config['training'][key] = str(step_id)
    config['training']['best_test_loss'] = str(t_loss)
    return t_loss


def _final_test_message(t_loss, best_test_loss):
    if t_loss <= best_test_loss:
        print("The last model is the best model.")
    else:
        print("Final test loss was not better than the best model.")
        print("Final Test Loss: {}".format(t_loss))
        print("Best Test Loss: {}".format(best_test_loss))


def _with_next(iterable):
    """(item, next item or None) pairs: the device-side analogue of a prefetching DataLoader - the step functions
    gather the next batch on their background stream while the current step's GEMMs run."""
    it = iter(iterable)
    try:
        cur = next(it)
    except StopIteration:
        return
    for nxt in it:
        yield cur, nxt
        cur = nxt
    yield cur, None


def _flush_losses(writer, pending, print_fmt=None, world=1):
    """Read back a block of per-batch losses (device scalars) with one sync and log them under the reference's tag.
    Entries are (step id, loss) or, when clipping, (step id, loss, gradient norm): the norms come back in the same
    copy and are logged as 'Grad Norm'."""
    if not pending:
        return 0.0
    norms = [e[2] for e in pending if len(e) > 2]
    got = torch.stack([e[1] for e in pending] + norms).cpu().tolist()
    vals, norm_vals = got[:len(pending)], got[len(pending):]
    if world > 1:
        rdist.check_health(pending[0][1].device)   # a rank that dropped out of the gradient exchange: fail loudly
    for i, (e, v) in enumerate(zip(pending, vals)):
        step_id = e[0]
        writer.add_scalar('Loss/Batch', v, step_id)
        if norm_vals:
            writer.add_scalar('Grad Norm', norm_vals[i], step_id)
        if print_fmt:
            print(print_fmt.format(step_id, v))
    pending.clear()
    return float(sum(vals))


# ---------------------------------------------------------------------------------------------------- train.py
def run_epoch_trainer(argv=None):
    config = _read_config(argv)
    sampling_rate = config['audio'].getint('sampling_rate')
    hop_length = config['audio'].getint('hop_length')
    segment_length = config['audio'].getint('segment_length')
    dataset = Path(config['dataset'].get('datapath'))
    if not dataset.exists():
        raise FileNotFoundError(dataset.resolve())
    my_audio = dataset / 'audio'
    test_audio = config['dataset'].get('test_dataset')
    dataset_test_audio = dataset / test_audio
    if not dataset_test_audio.exists():
        raise FileNotFoundError(dataset_test_audio.resolve())
    generate_test = config['dataset'].getboolean('generate_test')
    epochs = config['training'].getint('epochs')
    learning_rate = config['training'].getfloat('learning_rate')
    batch_size = config['training'].getint('batch_size')
    checkpoint_interval = config['training'].getint('checkpoint_interval')
    save_best_model_after = config['training'].getint('save_best_model_after')
    log_interval = config['training'].getint('log_interval', fallback=64)   # batches per loss read-back
    latent_dim = config['VAE'].getint('latent_dim')
    n_units = config['VAE'].getint('n_units')
    kl_beta = config['VAE'].getfloat('kl_beta')
    test_loss = _test_loss_enabled(config)
    max_grad_norm = _max_grad_norm(config)
    ema_decay = _ema_decay(config)
    deterministic = _deterministic(config)
    _apply_seed(_seed(config))
    start_time = time.time()
    config['extra']['start'] = time.asctime(time.localtime(start_time))

    rank, world, device = _common_setup(config)
    workdir = _make_workspace(config, dataset, rank)

    print('creating the dataset...')
    chunks = [audio_io.load_mono(f, sampling_rate)[0] for f in sorted(my_audio.glob('*.wav'))]
    if not chunks:
        raise FileNotFoundError("no .wav files in {}".format(my_audio))
    training_array = np.concatenate(chunks, axis=0)
    total_frames = len(training_array) // segment_length
    print('Total number of audio frames: {}'.format(total_frames))
    config['dataset']['total_frames'] = str(total_frames)
    training_dataset = AudioDataset(training_array, segment_length=segment_length, sampling_rate=sampling_rate,
                                    hop_size=hop_length, transform=ToTensor())
    loader = training_dataset.gpu_loader(batch_size, shuffle=True, device=device)
    loader.rank, loader.world = rank, world
    schedule = _schedule(config, _epoch_trainer_steps(config, len(training_dataset), world))

    writer = _NullWriter()
    if rank == 0:
        print("saving initial configs...")
        config_path = workdir / 'config.ini'
        with open(config_path, 'w') as configfile:
            config.write(configfile)
        checkpoint_dir = workdir / 'model' / 'checkpoints'
        os.makedirs(checkpoint_dir, exist_ok=True)
        log_dir = workdir / 'logs'
        os.makedirs(log_dir, exist_ok=True)
        writer = _summary_writer(log_dir, True)
        if generate_test:
            test_dataset, audio_log_dir = init_test_audio(workdir, test_audio, dataset_test_audio, sampling_rate,
                                                          segment_length)

    model = VAE(segment_length, n_units, latent_dim, precision=_precision(config)).to(device)
    optimizer = Adam(model.parameters(), lr=learning_rate)
    use_graph = config['training'].getboolean('cuda_graph', fallback=True)
    ring = max(64, log_interval)
    ema = ExponentialMovingAverage(model, ema_decay) if ema_decay is not None else None
    served = ema.module if ema is not None else model   # the weights that are evaluated, listened to and saved
    if world > 1:
        step = rdist.DataParallelTrainStep(model, optimizer, kl_beta, ring=ring, graph=use_graph, schedule=schedule,
                                           max_grad_norm=max_grad_norm, deterministic=deterministic, ema=ema)
    else:
        step = FusedTrainStep(model, optimizer, kl_beta, ring=ring, graph=use_graph, schedule=schedule,
                              max_grad_norm=max_grad_norm, deterministic=deterministic, ema=ema)

    # parameter histograms on the GPU (rank 0 only): one launch + one small asynchronous copy per set
    hist = ParamHistogramLogger(model, writer) if rank == 0 else None

    train_loss_prev = 1000000
    best_loss = 1000000
    final_loss = 1000000
    best_test_loss = float('inf')
    batch_id = 0
    for epoch in range(epochs):
        print('Epoch {}/{}'.format(epoch, epochs - 1))
        print('-' * 10)
        model.train()
        train_loss = 0.0
        pending = []
        for b, (data, nxt) in enumerate(_with_next(loader)):
            if world > 1:  # the last batch of an epoch may be short: normalise by the true global batch size
                step.global_batch = min(batch_size, len(training_dataset) - b * batch_size)
            loss = step(data, next_data=nxt)   # the next batch is gathered in the background of this step
            pending.append((batch_id, loss) if max_grad_norm is None else (batch_id, loss, step.grad_norm))
            _log_hparams(writer, schedule, optimizer, kl_beta, batch_id)
            batch_id += 1
            if len(pending) >= log_interval:
                train_loss += _flush_losses(writer, pending, world=world)
                if hist is not None:
                    hist.flush()
        train_loss += _flush_losses(writer, pending, world=world)
        print('====> Epoch: {} - Total loss: {} - Average loss: {:.9f}'.format(
            epoch, train_loss, train_loss / len(training_dataset)))
        writer.add_scalar('Loss/train_total', train_loss, epoch)
        writer.add_scalar('Loss/train_average', train_loss / len(training_dataset), epoch)
        if hist is not None:
            hist.record(epoch)
            hist.flush()

        if rank == 0 and epoch % checkpoint_interval == 0 and epoch != 0:
            print('Checkpoint - Epoch {}'.format(epoch))
            hist.flush(wait=True)
            state = _with_ema({'epoch': epoch, 'state_dict': model.state_dict(),
                              'optimizer': optimizer.state_dict()}, ema)
            if generate_test:
                audio_out = audio_log_dir.joinpath('test_reconst_{:05d}.wav'.format(epoch))
                test_predictions_np = _reconstruct_test(served, test_dataset, batch_size, device)
                audio_io.write_wav(audio_out, test_predictions_np, sampling_rate)
                print('Audio examples generated: {}'.format(audio_out))
                writer.add_audio('Reconstructed Audio', test_predictions_np, epoch, sample_rate=sampling_rate)
            torch.save(state, checkpoint_dir.joinpath('ckpt_{:05d}'.format(epoch)))
            if test_loss:
                t_loss = _evaluate_test(served, test_dataset, kl_beta, batch_size, writer, epoch)
                if epoch > save_best_model_after:
                    best_test_loss = _keep_best_test(served, t_loss, best_test_loss, workdir, config, 'best_epoch', epoch)
            elif (train_loss < train_loss_prev) and (epoch > save_best_model_after):
                save_path = workdir.joinpath('model').joinpath('best_model.pt')
                torch.save(served, save_path)
                print('Epoch {:05d}: Saved {}'.format(epoch, save_path))
                config['training']['best_epoch'] = str(epoch)
                best_loss = train_loss
            elif train_loss > train_loss_prev:
                print("Average loss did not improve.")
        # rank 0 alone wrote histograms / checkpoints / test audio above: nobody runs ahead into the next epoch's
        # gradient exchanges until it is back (the exchange waits for minutes, but there is no reason to queue up)
        rdist.sync_ranks()
        final_loss = train_loss

    if rank == 0:
        hist.flush(wait=True)
        print('Last Checkpoint - Epoch {}'.format(epochs))
        state = _with_ema({'epoch': epochs, 'state_dict': model.state_dict(),
                          'optimizer': optimizer.state_dict()}, ema)
        if generate_test:
            audio_out = audio_log_dir.joinpath('test_reconst_{:05d}.wav'.format(epochs))
            test_predictions_np = _reconstruct_test(served, test_dataset, batch_size, device)
            audio_io.write_wav(audio_out, test_predictions_np, sampling_rate)
            print('Last Audio examples generated: {}'.format(audio_out))
            writer.add_audio('Reconstructed Audio', test_predictions_np, epochs, sample_rate=sampling_rate)
        torch.save(state, checkpoint_dir.joinpath('ckpt_{:05d}'.format(epochs)))
        if test_loss:
            t_loss = _evaluate_test(served, test_dataset, kl_beta, batch_size, writer, epochs)
            if epochs > save_best_model_after:
                best_test_loss = _keep_best_test(served, t_loss, best_test_loss, workdir, config, 'best_epoch', epochs)
            _final_test_message(t_loss, best_test_loss)
        elif final_loss > train_loss_prev:
            print("Final loss was not better than the last best model.")
            print("Final Loss: {}".format(final_loss))
            print("Best Loss: {}".format(best_loss))
        else:
            print("The last model is the best model.")
        save_path = workdir.joinpath('model').joinpath('last_model.pt')
        torch.save(served, save_path)
        print('Training Finished: Saved the last model')
        config['extra']['end'] = time.asctime(time.localtime(time.time()))
        config['extra']['time_elapsed'] = str(time.time() - start_time)
        with open(config_path, 'w') as configfile:
            config.write(configfile)
        writer.close()
    return 0


# ---------------------------------------------------------------------------------------------------- train_iterable.py
def run_stream_trainer(argv=None):
    config = _read_config(argv)
    sampling_rate = config['audio'].getint('sampling_rate')
    hop_length = config['audio'].getint('hop_length')
    segment_length = config['audio'].getint('segment_length')
    dataset = Path(config['dataset'].get('datapath'))
    if not dataset.exists():
        raise FileNotFoundError(dataset.resolve())
    my_audio = dataset / 'audio'
    test_audio = config['dataset'].get('test_dataset')
    dataset_test_audio = dataset / test_audio
    if not dataset_test_audio.exists():
        raise FileNotFoundError(dataset_test_audio.resolve())
    generate_test = config['dataset'].getboolean('generate_test')
    total_num_frames = config['training'].getint('total_num_frames')
    learning_rate = config['training'].getfloat('learning_rate')
    batch_size = config['training'].getint('batch_size')
    checkpoint_interval = config['training'].getint('checkpoint_interval')
    total_num_batches = _stream_trainer_steps(config)
    schedule = _schedule(config, total_num_batches)
    log_interval = config['training'].getint('log_interval', fallback=64)
    histogram_interval = config['training'].getint('histogram_interval', fallback=checkpoint_interval)
    latent_dim = config['VAE'].getint('latent_dim')
    n_units = config['VAE'].getint('n_units')
    kl_beta = config['VAE'].getfloat('kl_beta')
    test_loss = _test_loss_enabled(config)
    max_grad_norm = _max_grad_norm(config)
    ema_decay = _ema_decay(config)
    deterministic = _deterministic(config)
    seed = _seed(config)
    if segment_length != 1024:
        raise ValueError("the streaming dataset frames at 1024 samples (rawvae/dataset.py:66); segment_length "
                         "= {} is not supported by train_iterable.py".format(segment_length))
    _apply_seed(seed)
    start_time = time.time()
    config['extra']['start'] = time.asctime(time.localtime(start_time))

    rank, world, device = _common_setup(config)
    workdir = _make_workspace(config, dataset, rank)

    log_file, original_stdout = None, sys.stdout
    if rank == 0:
        console_log_path = workdir / 'console_log'
        log_file = open(console_log_path, 'w')
        sys.stdout = Tee(sys.stdout, log_file)
        print("Console logging started - all output will be saved to: {}".format(console_log_path))
    try:
        print('creating the dataset...')
        print('Found {} audio files'.format(len(list(my_audio.glob('*.wav')))))
        training_dataset = IterableAudioDataset(audio_folder=my_audio, sampling_rate=sampling_rate,
                                                hop_size=hop_length, dtype=torch.float32, device=device, shuffle=True)
        stream = training_dataset.gpu_stream(batch_size, device, pcm16="auto")
        stream.rank, stream.world = rank, world

        writer = _NullWriter()
        if rank == 0:
            print("saving initial configs...")
            config_path = workdir / 'config.ini'
            with open(config_path, 'w') as configfile:
                config.write(configfile)
            checkpoint_dir = workdir / 'model' / 'checkpoints'
            os.makedirs(checkpoint_dir, exist_ok=True)
            log_dir = workdir / 'logs'
            os.makedirs(log_dir, exist_ok=True)
            writer = _summary_writer(log_dir, True)
            if generate_test:
                test_dataset, audio_log_dir = init_test_audio(workdir, test_audio, dataset_test_audio, sampling_rate,
                                                              segment_length)

        model = VAE(segment_length, n_units, latent_dim, precision=_precision(config)).to(device)
        optimizer = Adam(model.parameters(), lr=learning_rate)
        use_graph = config['training'].getboolean('cuda_graph', fallback=True)
        ring = max(64, log_interval)
        ema = ExponentialMovingAverage(model, ema_decay) if ema_decay is not None else None
        served = ema.module if ema is not None else model   # the weights that are evaluated, listened to and saved
        if world > 1:
            step = rdist.DataParallelTrainStep(model, optimizer, kl_beta, global_batch=batch_size, ring=ring,
                                               graph=use_graph, schedule=schedule, max_grad_norm=max_grad_norm,
                                               deterministic=deterministic, ema=ema)
        else:
            step = FusedTrainStep(model, optimizer, kl_beta, ring=ring, graph=use_graph, schedule=schedule,
                                  max_grad_norm=max_grad_norm, deterministic=deterministic, ema=ema)

        hist = ParamHistogramLogger(model, writer) if rank == 0 and histogram_interval > 0 else None

        train_loss_prev = 1000000
        best_loss = 1000000
        best_test_loss = float('inf')
        model.train()
        train_loss = 0.0
        batch_id = 0
        pending = []
        fmt = '====> Batch: {} - Loss: {:.9f}'
        for data, nxt in _with_next(islice(stream, total_num_batches)):
            loss = step(data, next_data=nxt)   # the next batch is gathered in the background of this step
            pending.append((batch_id, loss) if max_grad_norm is None else (batch_id, loss, step.grad_norm))
            _log_hparams(writer, schedule, optimizer, kl_beta, batch_id)
            at_checkpoint = batch_id % checkpoint_interval == 0 and batch_id != 0
            if len(pending) >= log_interval or at_checkpoint:
                train_loss += _flush_losses(writer, pending, fmt if rank == 0 else None, world=world)
                if hist is not None:
                    hist.flush()
            if hist is not None and batch_id % histogram_interval == 0:
                hist.record(batch_id)   # same stream as the step: sees its Adam update, precedes the next step
            if rank == 0 and at_checkpoint:
                print('Checkpoint - Epoch {}'.format(batch_id))
                if hist is not None:
                    hist.flush(wait=True)
                state = _with_ema({'batch_id': batch_id, 'state_dict': model.state_dict(),
                                  'optimizer': optimizer.state_dict()}, ema)
                if generate_test:
                    audio_out = audio_log_dir.joinpath('test_reconst_{:05d}.wav'.format(batch_id))
                    test_predictions_np = _reconstruct_test(served, test_dataset, batch_size, device)
                    audio_io.write_wav(audio_out, test_predictions_np, sampling_rate)
                    print('Audio examples generated: {}'.format(audio_out))
                    writer.add_audio('Reconstructed Audio', test_predictions_np, batch_id, sample_rate=sampling_rate)
                torch.save(state, checkpoint_dir.joinpath('ckpt_{:05d}'.format(batch_id)))
                if test_loss:
                    t_loss = _evaluate_test(served, test_dataset, kl_beta, batch_size, writer, batch_id)
                    best_test_loss = _keep_best_test(served, t_loss, best_test_loss, workdir, config, 'best_model',
                                                     batch_id)
                elif train_loss < train_loss_prev:
                    save_path = workdir.joinpath('model').joinpath('best_model.pt')
                    torch.save(served, save_path)
                    print('batch_id {:05d}: Saved {}'.format(batch_id, save_path))
                    config['training']['best_model'] = str(batch_id)
                    best_loss = train_loss
                elif train_loss > train_loss_prev:
                    print("Loss did not improve.")
            if at_checkpoint or (histogram_interval > 0 and batch_id % histogram_interval == 0):
                rdist.sync_ranks()   # rank 0 alone did I/O above (same condition on every rank): wait for it
            batch_id += 1
        train_loss += _flush_losses(writer, pending, fmt if rank == 0 else None, world=world)
        final_loss = train_loss

        if rank == 0:
            if hist is not None:
                hist.flush(wait=True)
            print('Last Checkpoint - batch_id {}'.format(batch_id))
            state = _with_ema({'batch_id': batch_id, 'state_dict': model.state_dict(),
                              'optimizer': optimizer.state_dict()}, ema)
            if generate_test:
                audio_out = audio_log_dir.joinpath('test_reconst_{:05d}.wav'.format(total_num_batches))
                test_predictions_np = _reconstruct_test(served, test_dataset, batch_size, device)
                audio_io.write_wav(audio_out, test_predictions_np, sampling_rate)
                print('Last Audio examples generated: {}'.format(audio_out))
                writer.add_audio('Reconstructed Audio', test_predictions_np, batch_id, sample_rate=sampling_rate)
            torch.save(state, checkpoint_dir.joinpath('ckpt_{:05d}'.format(total_num_batches)))
            if test_loss:
                t_loss = _evaluate_test(served, test_dataset, kl_beta, batch_size, writer, batch_id)
                best_test_loss = _keep_best_test(served, t_loss, best_test_loss, workdir, config, 'best_model',
                                                 total_num_batches)
                _final_test_message(t_loss, best_test_loss)
            elif train_loss > train_loss_prev:
                print("Final loss was not better than the last best model.")
                print("Final Loss: {}".format(final_loss))
                print("Best Loss: {}".format(best_loss))
            else:
                print("The last model is the best model.")
            save_path = workdir.joinpath('model').joinpath('last_model.pt')
            torch.save(served, save_path)
            print('Training Finished: Saved the last model')
            config['extra']['end'] = time.asctime(time.localtime(time.time()))
            config['extra']['time_elapsed'] = str(time.time() - start_time)
            with open(config_path, 'w') as configfile:
                config.write(configfile)
            writer.close()
    finally:
        if log_file is not None:
            sys.stdout = original_stdout
            log_file.close()
            print("Training completed. Console log saved to: {}".format(console_log_path))
    return 0
