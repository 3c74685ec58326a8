#!/usr/bin/env python
"""Benchmark of the hot path: training frames/sec (forward + loss + backward + Adam) of the default.ini VAE
(S=1024, H=2048, L=256) on synthetic 44.1 kHz sine+noise audio, 8192 frames per GPU per step (BASELINE.json
configs[1]; weak scaling for N > 1).

    python bench.py --gpus N --steps K --warmup W            # our arm (sm_100a kernels)
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU (oracle port)

Prints ONE JSON line on rank 0. See DESIGN.md "Measurement" for what each key means.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

S, H, L = 1024, 2048, 256            # default.ini:5,18-19
HOP = 128                            # default.ini:4
KL_BETA, LR = 1e-4, 1e-4             # default.ini:20,26
BATCH = 8192                         # BASELINE.json configs[1]
SR = 44100
FLOP_PER_FRAME = 30408704            # SURVEY.md 8(d): fwd + bwd GEMMs only (no fc1 dgrad)
WORKLOAD = "default.ini VAE (S=1024,H=2048,L=256) bf16 training, batch 8192 frames/GPU, synthetic 44.1 kHz sine+noise audio"


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"bf16_burst": d.get("bf16_tflops"), "bf16_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "measured"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


def synth_wav(rng: np.random.Generator, n_samples: int, sr: int = SR) -> np.ndarray:
    """SURVEY.md 8(d): 0.5*sin(2*pi*f*t + phi) + 0.05*N(0,1), f log-uniform in [55, 7040] Hz, clipped, as the float32
    value of 16-bit PCM (int16 / 32768). Same formula as the tests' generator; restated here so that the GPU arm
    of the bench imports nothing from oracle/."""
    f = math.exp(rng.uniform(math.log(55.0), math.log(7040.0)))
    phi = rng.uniform(0, 2 * math.pi)
    t = np.arange(n_samples) / sr
    x = 0.5 * np.sin(2 * math.pi * f * t + phi) + 0.05 * rng.standard_normal(n_samples)
    pcm = np.clip(np.round(x * 32767.0), -32768, 32767).astype(np.int16)
    return (pcm.astype(np.float32) / 32768.0).astype(np.float32)


def synth_corpus(n_files: int, seconds: float, seed: int = 1234) -> np.ndarray:
    """SURVEY.md 8(d) synthetic wav folder, concatenated as train.py:118-126 does: float32 = int16 PCM / 32768."""
    rng = np.random.default_rng(seed)
    return np.concatenate([synth_wav(rng, int(seconds * SR), SR) for _ in range(n_files)])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------- CPU arm
def cpu_train_steps(n_steps: int, warmup: int, threads: int, frames: int = BATCH):
    """The reference's training-loop body (train_iterable.py:200-210) restated by the oracle port, fp32, torch CPU
    with all host threads - i.e. the same ATen kernels the reference's own CPU path runs. Returns per-step seconds."""
    from oracle import rawvae_oracle as O
    torch.set_num_threads(threads)
    p = O.init_params(S, H, L, seed=0)
    st = O.adam_init(p)
    gen = torch.Generator().manual_seed(1)
    x = torch.rand(frames, S, generator=gen) * 2 - 1
    times = []
    for i in range(warmup + n_steps):
        eps = torch.randn(frames, L, generator=gen)
        t0 = time.perf_counter()
        O.train_step(p, st, x, eps, KL_BETA, LR)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return times


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    # bounded sample: a step is a full 8192-frame batch when the whole run fits ~150 s, else a smaller batch
    probe = cpu_train_steps(1, 1, threads)[0]
    frames = BATCH
    budget = 150.0
    while frames > 512 and probe * (frames / BATCH) * (args.steps + args.warmup) > budget:
        frames //= 2
    times = cpu_train_steps(args.steps, args.warmup, threads, frames)
    total = sum(times)
    fps = frames * len(times) / total
    out = {
        "impl": "reference", "metric": "train frames/sec (fwd+bwd+Adam)", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_step": frames, "device": "host CPU"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"{len(times)} training steps of {frames} frames each, oracle port (torch CPU fp32, "
                                   f"{threads} threads, {total:.1f} s)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------------- GPU arm
class NvmlSampler:
    """SM clock / clocks-event reasons DURING the timed region, polled through NVML every few milliseconds by a
    thread (nvidia-smi -lms cannot sample faster than ~100 ms, longer than a 20-step block). Falls back to the
    nvidia-smi sampler when NVML is unavailable."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
               (0x4, "sw_power_cap"))

    def __init__(self, dev: torch.device, period_s: float = 0.005):
        self.period, self.samples, self.bits, self.h, self.nv = period_s, [], 0, None, None
        self.fallback = None
        try:
            import pynvml
            pynvml.nvmlInit()
            props = torch.cuda.get_device_properties(dev)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(props.uuid)).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(dev.index or 0)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None
            self.fallback = ClockSampler(dev.index or 0)

    def _loop(self):
        nv = self.nv
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.bits |= int(reasons_fn(self.h))
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.h is None:
            return self.fallback.start()
        self._stop = threading.Event()
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def stop(self):
        if self.h is None:
            return self.fallback.stop()
        self._stop.set()
        self.t.join(timeout=1.0)
        sm = self.samples
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": float(min(sm)) if sm else None,
                "sm_max_mhz": self.max_mhz, "reasons": [n for b, n in self.REASONS if self.bits & b],
                "samples": len(sm), "source": "nvml, polled during the timed blocks"}


MOMENT_SAMPLE = 1 << 20              # Adam moments dumped per buffer (of 5.77 M): keeps a dump near 32 MB


def dump_outputs(out_dir: str, model, opt, loss: torch.Tensor) -> None:
    """What a caller of the timed step holds after its last call, as float32 .npy files in out_dir: `loss.npy` (the
    step's return value), `<parameter name>.npy` (every updated weight and bias, in full) and
    `exp_avg.sample.npy` / `exp_avg_sq.sample.npy` (the optimizer's moments over all parameters in named_parameters()
    order, at a fixed seeded sample of MOMENT_SAMPLE positions). The inputs of a run depend on the arguments only, so
    two builds run with the same arguments can be compared file by file. Two runs of one build agree to rounding,
    not bit for bit: split-K partial products are summed in arrival order, and Adam turns a rounding difference in a
    near-zero gradient into up to one learning-rate step of a weight."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().float().cpu().numpy()}
    named = list(model.named_parameters())
    for name, p in named:
        arrays[name] = p.detach().float().cpu().numpy()
    idx = np.sort(np.random.default_rng(0).choice(sum(p.numel() for _, p in named), MOMENT_SAMPLE, replace=False))
    for key in ("exp_avg", "exp_avg_sq"):
        flat = torch.cat([opt.state[p][key].detach().float().flatten() for _, p in named]).cpu().numpy()
        arrays[key + ".sample"] = flat[idx]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    from rawaudiovae_kelsey_b200 import dist as rdist
    from rawaudiovae_kelsey_b200 import ops
    from rawaudiovae_kelsey_b200.model import FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from rawvae.model import VAE
    import torch.distributed as dist

    rank, world, local_rank = rdist.init_from_env("nccl")
    if world != args.gpus and rank == 0 and world > 1:
        print(f"# note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    peaks = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # model + optimizer (random init of the default.ini architecture)
    torch.manual_seed(0)
    model = VAE(S, H, L, precision=args.precision).to(dev)
    model.eps_seed = 1
    opt = Adam(model.parameters(), lr=LR)
    if world > 1:
        step_fn = rdist.DataParallelTrainStep(model, opt, KL_BETA, global_batch=BATCH * world, graph=args.graph)
    else:
        step_fn = FusedTrainStep(model, opt, KL_BETA, graph=args.graph)

    # synthetic corpus resident in HBM (every rank holds it; rank r draws its own frame indices)
    corpus = synth_corpus(args.files, args.seconds)
    from rawaudiovae_kelsey_b200.dataset import resident_audio
    audio = resident_audio(corpus, dev)     # the product's loader path: 16-bit PCM content stays int16 in HBM (lossless)
    n_frames = (len(corpus) + HOP - 1) // HOP - S // HOP + 1

    # Steady state before anything is timed. A CUDA-graph step function captures one graph per input signature after
    # one eager call of that signature, and the pipelined signature contains the parity of the plan's double-buffered
    # input set: eager, eager, capture, capture, then replays. The untimed pre-steps therefore run for at least
    # --warmup steps AND until NEED consecutive steps were plain replays; the timed blocks assert that no capture and
    # no eager step happened inside them. Each leg then runs one untimed lead-in block of --steps steps, shaped like a
    # timed block and with the clock sampler already running: on a B200 (1000 W) a block timed straight after the
    # set-up work measured ~2 % slower than every block after it.
    NEED = 4
    pre_steps = max(args.warmup, 2 * step_fn.graph_warmup + 2 + NEED) if args.graph else args.warmup
    est_ms = 0.35 if args.precision == "bf16" else 1.0
    # Statistic. Every timed block is EXACTLY --steps steps between barrier + synchronize, and a leg is --blocks blocks
    # (default 1), so `value` and `e2e` time exactly --steps steps each unless --blocks asks for more; with several
    # blocks they are the median block. A short run is at boost clocks. With --sustained each leg then simply keeps
    # going for sus_blocks more blocks (~0.4 s of continuous load): ~100 ms in, the board's power cap starts to pull the
    # SM clock of a single busy GPU down, and it keeps drifting for seconds (under data parallelism the GPUs idle in the
    # exchange and stay at boost). The median of the second half of those later blocks is reported as `sustained` -
    # what a long job sees early on - and is never mixed into `value`.
    n_blocks = max(1, args.blocks)
    sus_blocks = int(min(200, math.ceil(400.0 / (args.steps * est_ms)))) if args.sustained else 0

    def leg_stats(all_ms):
        """(median ms per block of the first n_blocks blocks, median of the second half of the later blocks or None)"""
        if sus_blocks == 0:
            return float(np.median(all_ms)), None
        rest = all_ms[n_blocks:]
        return float(np.median(all_ms[:n_blocks])), float(np.median(rest[len(rest) // 2:]))

    # batch i = a fresh random 8192-frame gather; a pool of index sets is cycled (the pool's footprint is far larger
    # than L2). Step i also hands the step function batch i + 1, which it gathers (and draws the noise for) on its
    # background stream while the GEMMs of step i run - the device-side analogue of a prefetching DataLoader.
    pool = min(256, pre_steps + (1 + n_blocks + sus_blocks) * args.steps + 1)
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    frame_idx = torch.randint(0, n_frames, (pool, BATCH), generator=g, device=dev, dtype=torch.int64)
    batches = [FrameBatch(audio, BATCH, HOP, S, frame_idx=frame_idx[i]) for i in range(pool)]

    def device_step(i):
        nxt = batches[(i + 1) % pool] if args.prefetch else None
        return step_fn(batches[i % pool], next_data=nxt)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def settle(step_once, i):
        """untimed pre-steps; returns the next step index"""
        for _ in range(pre_steps):
            step_once(i)
            i += 1
        if args.graph and step_fn.steady < NEED:
            raise RuntimeError(f"graph replay not steady after {pre_steps} pre-steps: {step_fn.stats}")
        return i

    def timed_blocks(step_once, i, end_of_block=None, blocks=None):
        """n_blocks blocks of EXACTLY --steps steps, each bracketed by barrier + synchronize; block times are the
        max over ranks. Returns (block ms list, next step index, last loss, stats delta)."""
        s0 = dict(step_fn.stats)
        times, loss = [], None
        for _ in range(blocks or n_blocks):
            barrier()
            e0.record()
            for _ in range(args.steps):
                loss = step_once(i)
                i += 1
            if end_of_block is not None:
                end_of_block()
            e1.record()
            barrier()
            times.append(e0.elapsed_time(e1))
        t = torch.tensor(times, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        delta = {k: step_fn.stats[k] - s0[k] for k in s0}
        return [float(v) for v in t.cpu()], i, loss, delta

    # ---- value: inputs resident in HBM, whole step = framing + fwd + loss + bwd (+ allreduce) + Adam
    i = settle(device_step, 0)
    barrier()
    if world > 1:   # data parallelism kept the replicas bit-identical through the pre-steps (checked once, untimed)
        ref_params = model._flat.params.clone()
        dist.broadcast(ref_params, src=0)
        same = torch.tensor([int(torch.equal(ref_params, model._flat.params))], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        assert int(same) == 1, "data-parallel replicas diverged"
        del ref_params
    clocks = NvmlSampler(dev)
    if rank == 0:
        clocks.start()
    _, i, _, _ = timed_blocks(device_step, i, blocks=1)     # lead-in block, untimed
    l0 = ops.launch_count(dev) + step_fn.replayed_launches
    block_ms, i, loss, delta = timed_blocks(device_step, i, blocks=n_blocks)
    launches = ops.launch_count(dev) + step_fn.replayed_launches - l0   # eager launches + kernels inside graph replays
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, opt, loss)
    sus_clk = None
    if sus_blocks > 0:   # the leg simply continues (no gap beyond the per-block barrier); clocks sampled separately
        sclocks = NvmlSampler(dev)
        if rank == 0:
            sclocks.start()
        later_ms, i, loss, d2 = timed_blocks(device_step, i, blocks=sus_blocks)
        sus_clk = sclocks.stop() if rank == 0 else None
        block_ms = block_ms + later_ms
        delta = {k: delta[k] + d2[k] for k in delta}
    last_loss = float(loss)
    ms, sus_ms = leg_stats(block_ms)
    value = BATCH * world * args.steps / (ms * 1e-3)
    if args.graph:
        assert delta["captures"] == 0 and delta["eager"] == 0, f"capture / eager step inside the timed region: {delta}"

    # ---- e2e: HOST buffers. Every step the host supplies the next chunk of the wav stream from pinned memory
    # (train_iterable.py's streaming pattern: 8192 consecutive frames at hop 128 = 1 049 472 samples), the GPU
    # frames it, trains on it, and the step's loss is read back to pinned host memory.
    chunk = (BATCH - 1) * HOP + S
    n_chunks = max(1, (len(corpus) - chunk) // (BATCH * HOP))
    host_audio = torch.from_numpy(corpus).pin_memory()
    n_e2e = pre_steps + (1 + n_blocks + sus_blocks) * args.steps
    host_loss = torch.zeros(n_e2e, dtype=torch.float32).pin_memory()
    dbuf = [torch.empty(chunk, dtype=torch.float32, device=dev) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)     # loss read-back: off the compute stream, so it never delays a step
    step_done = [torch.cuda.Event() for _ in range(4)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    main = torch.cuda.current_stream()

    def issue_copy(j):
        """chunk j of the wav stream: pinned host memory -> dbuf[j % 2] on the copy stream"""
        b = j % 2
        off = ((j * world + rank) % n_chunks) * BATCH * HOP
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[b])
            dbuf[b].copy_(host_audio[off:off + chunk], non_blocking=True)       # H2D from pinned memory
            ready[b].record(copy_stream)
        main.wait_event(ready[b])
        return FrameBatch(dbuf[b], BATCH, HOP, S, first_frame=0)

    pending = {}

    def e2e_step(j):
        cur = pending.pop(j, None) or issue_copy(j)
        nxt = None
        if args.prefetch:
            nxt = pending[j + 1] = issue_copy(j + 1)     # its frames are gathered in the background of step j
        loss = step_fn(cur, next_data=nxt)
        freed[(j + 1) % 2 if nxt is not None else j % 2].record(main)           # that buffer has been gathered
        ev = step_done[j % 4]
        ev.record(main)
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(ev)
            host_loss[j % n_e2e].copy_(loss, non_blocking=True)                 # D2H read of the step's result
        return loss

    for b in range(2):
        freed[b].record(main)
    j = settle(e2e_step, 0)
    # a block ends when its last loss has reached the host buffer
    loss_on_host = lambda: main.wait_stream(d2h_stream)
    _, j, _, _ = timed_blocks(e2e_step, j, end_of_block=loss_on_host, blocks=1)     # lead-in block, untimed
    e2e_block_ms, j, _, e2e_delta = timed_blocks(e2e_step, j, end_of_block=loss_on_host,
                                                 blocks=n_blocks + sus_blocks)
    e2e_ms, e2e_sus_ms = leg_stats(e2e_block_ms)
    e2e_value = BATCH * world * args.steps / (e2e_ms * 1e-3)
    torch.cuda.synchronize()
    assert np.isfinite(host_loss.numpy()).all()
    if args.graph:
        assert e2e_delta["captures"] == 0 and e2e_delta["eager"] == 0, f"capture / eager step in the e2e region: {e2e_delta}"

    # ---- roofline of the dominant kernel family (tcgen05 GEMMs), timed live with CUDA events on the launch stream
    roofline, breakdown = None, None
    if rank == 0:
        plan = model._plan_for(BATCH)
        plan.enable_timing(True)
        nroof = min(args.steps, 20)
        local_step = FusedTrainStep(model, opt, KL_BETA)   # no collectives: only rank 0 runs this attribution pass
        for k in range(nroof):
            local_step(batches[k % pool])
        torch.cuda.synchronize()
        tm_all = plan.read_timing()
        plan.enable_timing(False)
        tm = {k: v for k, v in tm_all.items() if k in plan.GEMM_SLOTS}
        aux = {k: 1e3 * v[0] / nroof for k, v in tm_all.items() if k in plan.AUX_SLOTS and v[1] > 0}
        gemm_ms = sum(v[0] for v in tm.values()) / nroof
        flops = sum(v[1] * v[2] for v in tm.values()) / nroof
        passes = 3 if args.precision == "fp32" else 1
        achieved = flops / (gemm_ms * 1e-3) / 1e12
        # the attribution pass runs the step's OWN launches (the fused dgrad + weight-gradient launches included, their
        # flops booked together) one at a time: events around each launch serialise the stream (no overlap of a kernel's
        # prologue with its predecessor's tail, no background stream), ~6 ms in total: a burst measurement, so the
        # denominator is the measured burst peak
        peak = peaks["bf16_burst"]
        traffic, traffic_src = None, None
        for name in ("r2_gemms_ncu.json", "r1_gemms_ncu.json"):   # dram__bytes_read + write of the 11 GEMMs, one ncu capture
            ncu_json = ROOT / "profiles" / name
            if ncu_json.exists() and args.precision == "bf16":
                try:
                    traffic = float(json.loads(ncu_json.read_text())["dram_bytes_per_step"])
                    traffic_src = f"profiles/{name} (ncu --set full, sum over the 11 GEMM launches of a step)"
                    break
                except Exception:
                    traffic = None
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "kernel": "rvae::gemm_kernel<*> / gemm_chain_kernel_2cta<*>: the 11 GEMMs of a step in the 9 launches the step "
                              "uses (stages 0 and 2 of backward: dgrad + weight gradient fused into one launch)",
                    "launches_per_step": sum(v[1] for v in tm.values()) / nroof,
                    "peak_kind": f"bf16_tflops burst ({peaks['source']}): each launch timed alone",
                    "algorithmic_flops_per_step": flops, "gemm_ms_per_step": gemm_ms,
                    "tensor_passes": passes}
        fused_with = {"B4d": "B4w", "B2d": "B2w", "B3d": "B3w"}   # a fused launch is booked on the dgrad's slot
        label = lambda k: f"{k}+{fused_with[k]}" if k in fused_with and tm.get(fused_with[k], (0, 0, 0))[1] == 0 else k
        breakdown = {label(k): {"us": 1e3 * v[0] / max(v[1], 1), "tflops": (v[2] / (v[0] / max(v[1], 1) * 1e-3) / 1e12)
                                if v[0] > 0 else None} for k, v in tm.items() if v[1] > 0}
        breakdown["other_kernels_us_per_step"] = aux

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload on the host cores
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        t1 = cpu_train_steps(1, 1, threads)[0]
        n = int(min(30, max(3, round(15.0 / max(t1, 1e-3)))))
        times = cpu_train_steps(n, 0, threads)
        cpu_baseline = {"value": BATCH * len(times) / sum(times), "unit": "frames/s", "cores": threads, "kind": "port",
                        "sample": f"{len(times)} full {BATCH}-frame training steps of the oracle port "
                                  f"(torch CPU fp32, {threads} threads, {sum(times):.1f} s)"}

    # ---- the other BASELINE.json configs (N = 1 only): extra keys of the same line
    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        extras = extra_legs(dev, audio, n_frames, peaks)

    exchange = None
    if world > 1:
        from rawaudiovae_kelsey_b200 import _lib as rlib
        mc = bool(rlib.load().rvae_dp_uses_multicast(ops.ctx(dev)))
        exchange = ("own all-reduce kernel, in-switch reduction over an NVLS multicast mapping (multimem.ld_reduce / multimem.st)"
                    if mc else ("NCCL all-reduce" if os.environ.get("RVAE_DP_BACKEND", "auto") == "nccl"
                                else "own all-reduce kernel over NVLink peer memory (peer loads + posted peer writes)"))
    if rank == 0:
        ms_per_step = ms / args.steps
        whole_tflops = value * FLOP_PER_FRAME / world / 1e12
        sustained = None
        if sus_ms is not None:
            sustained = {"value": BATCH * world * args.steps / (sus_ms * 1e-3), "unit": "frames/s",
                         "ms_per_step": sus_ms / args.steps, "blocks": sus_blocks,
                         "e2e_value": BATCH * world * args.steps / (e2e_sus_ms * 1e-3), "clocks": sus_clk,
                         "statistic": "median of the second half of the blocks that follow the first %d of each leg "
                                      "(continuous load for ~0.4 s; on one GPU the power cap is acting and still "
                                      "drifting)" % n_blocks}
        out = {
            "metric": "train frames/sec (fwd+bwd+Adam)", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": BATCH, "global_batch": BATCH * world, "hop": HOP,
                       "precision": args.precision, "parallelism": f"dp{world}", "exchange": exchange, "cuda_graph": bool(args.graph), "prefetch_next_batch": bool(args.prefetch),
                       "l2": "per-step working set ~330 MB (activations + weights + moments) exceeds the 126 MB L2; "
                             "a different random 8192-frame gather from a %.0f MB corpus (%s in HBM) every step"
                             % (audio.numel() * audio.element_size() / 1e6, "16-bit PCM, lossless" if audio.dtype == torch.int16 else "float32"),
                       "corpus": f"{args.files} files x {args.seconds:.0f} s, 0.5*sin+0.05*noise, rng 1234"},
            "timing": {"blocks": n_blocks, "steps_per_block": args.steps,
                       "statistic": "median of the %d timed blocks of the leg; max over ranks per block" % n_blocks,
                       "later_blocks_for_sustained": sus_blocks,
                       "pre_steps_untimed": pre_steps, "lead_in_steps_untimed": args.steps, "block_ms": [round(v, 4) for v in block_ms],
                       "captures_in_timed_region": delta["captures"], "eager_steps_in_timed_region": delta["eager"],
                       "graph_replays_in_timed_region": delta["replays"],
                       "e2e_block_ms": [round(v, 4) for v in e2e_block_ms],
                       "e2e_captures_in_timed_region": e2e_delta["captures"],
                       "e2e_eager_steps_in_timed_region": e2e_delta["eager"]},
            "final_loss": last_loss,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": chunk * 4, "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / args.steps,
                    "path": "pinned host wav-stream chunk -> H2D -> FusedTrainStep(FrameBatch) -> loss D2H; the chunk's 8192 frames "
                            "are consecutive (train_iterable.py's stream) and therefore read in place - no gather kernel, "
                            "which is why e2e can exceed `value` (random 8192-frame gather from the resident corpus)"},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": roofline,
            # whole step (framing, loss, Adam, all-reduce included) per GPU, like with like: `value` (a short run at boost
            # clocks) against the burst peak, the later blocks against the sustained peak (a 4 s matmul run)
            "roofline_whole_step": {"bound": "tensor", "achieved": whole_tflops, "peak": peaks["bf16_burst"],
                                    "unit": "TFLOP/s", "frac": whole_tflops / peaks["bf16_burst"],
                                    "peak_kind": f"bf16_tflops burst ({peaks['source']}): `value` is a {n_blocks * args.steps}-step run",
                                    "sustained_achieved": sustained and sustained["value"] * FLOP_PER_FRAME / world / 1e12,
                                    "sustained_peak": peaks["bf16_sustained"],
                                    "sustained_frac": sustained and sustained["value"] * FLOP_PER_FRAME / world / 1e12 / peaks["bf16_sustained"]},
            "sustained": sustained,
            "gemm_breakdown": breakdown,
            "cpu_baseline": cpu_baseline,
        }
        if extras:
            out.update(extras)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# ----------------------------------------------------------------------------------------------------- other configs
def _median_blocks(step_once, n_blocks, steps, i0=0):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out, i = [], i0
    for _ in range(n_blocks):
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            step_once(i)
            i += 1
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return float(np.median(out)), out, i


def leg_fp32_mode(dev, audio, n_frames, peaks):
    """default.ini VAE, B = 8192, fp32 mode: every GEMM as 3 tensor-core passes over split-bf16 operands into one fp32
    TMEM accumulator (~2^-16 relative; the north star's "fp32-mode within 1e-4")."""
    from rawaudiovae_kelsey_b200.model import FrameBatch, FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from rawvae.model import VAE
    torch.manual_seed(0)
    model = VAE(S, H, L, precision="fp32").to(dev)
    model.eps_seed = 1
    step_fn = FusedTrainStep(model, Adam(model.parameters(), lr=LR), KL_BETA, graph=True)
    g = torch.Generator(device=dev).manual_seed(7)
    pool = 32
    idx = torch.randint(0, n_frames, (pool, BATCH), generator=g, device=dev, dtype=torch.int64)
    fbs = [FrameBatch(audio, BATCH, HOP, S, frame_idx=idx[k]) for k in range(pool)]
    once = lambda i: step_fn(fbs[i % pool], next_data=fbs[(i + 1) % pool])
    for i in range(10):
        once(i)
    assert step_fn.steady >= 4, step_fn.stats
    s0 = dict(step_fn.stats)
    ms, blocks, _ = _median_blocks(once, 5, 20, 10)
    assert step_fn.stats["captures"] == s0["captures"] and step_fn.stats["eager"] == s0["eager"]
    fps = BATCH * 20 / (ms * 1e-3)
    alg = fps * FLOP_PER_FRAME / 1e12
    return {"workload": "default.ini VAE fp32 mode (3-pass split-bf16), batch 8192, whole training step",
            "value": fps, "unit": "frames/s", "ms_per_step": ms / 20, "block_ms": [round(v, 3) for v in blocks],
            "roofline": {"bound": "tensor", "achieved": 3 * alg, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                         "frac": 3 * alg / peaks["bf16_sustained"], "algorithmic_tflops": alg, "tensor_passes": 3,
                         "peak_kind": f"bf16_tflops_sustained ({peaks['source']}), executed tensor flops = 3 x algorithmic"}}


def leg_stream_4096(dev, peaks):
    """kelsey_iterable.ini pattern (BASELINE.json configs[3]): batch 4096, frames of long wav streams framed on the GPU.
    END TO END from wav files on disk: a worker thread decodes PCM16 files into pinned memory, they are copied into a
    device ring smaller than the corpus (so every cycle re-uploads: the streaming case), batches straddle files."""
    import tempfile
    import scipy.io.wavfile as wavfile
    from rawaudiovae_kelsey_b200.dataset import IterableAudioDataset
    from rawaudiovae_kelsey_b200.model import FusedTrainStep
    from rawaudiovae_kelsey_b200.optim import Adam
    from rawaudiovae_kelsey_b200.trainer import _with_next
    from rawvae.model import VAE
    B4, n_files, secs = 4096, 4, 300.0      # long streams (SURVEY.md 8d: config 4 frames 10-minute files)
    with tempfile.TemporaryDirectory() as tmp:
        rng = np.random.default_rng(4321)
        base = synth_wav(rng, int(30.0 * SR), SR)
        for k in range(n_files):    # each file: ten differently rotated copies of a 30 s sine+noise clip (cheap to make)
            x = np.concatenate([np.roll(base, 7919 * (10 * k + j)) for j in range(int(secs / 30.0))])
            wavfile.write(os.path.join(tmp, f"stream{k}.wav"), SR, np.round(x * 32768.0).clip(-32768, 32767).astype(np.int16))
        ds = IterableAudioDataset(tmp, SR, HOP, torch.float32, dev, shuffle=True)
        file_bytes = int(secs * SR) * 2
        stream = ds.gpu_stream(B4, dev, pcm16=True, cache_bytes=int(2.5 * file_bytes))
        torch.manual_seed(0)
        model = VAE(S, H, L).to(dev)
        model.eps_seed = 1
        step_fn = FusedTrainStep(model, Adam(model.parameters(), lr=LR), KL_BETA, graph=True)
        pairs = _with_next(iter(stream))
        once = lambda i: _stream_step(step_fn, pairs)
        for i in range(80):     # past a file boundary: both input layouts (run read in place / gathered straddler) captured
            once(i)
        s0 = dict(step_fn.stats)
        up0 = dict(stream.stats)
        ms, blocks, _ = _median_blocks(once, 7, 40, 80)
        d = {k: step_fn.stats[k] - s0[k] for k in s0}
        fps = B4 * 40 / (ms * 1e-3)
        uploaded = stream.stats["bytes_uploaded"] - up0["bytes_uploaded"]
        return {"workload": "kelsey_iterable.ini pattern: default.ini VAE bf16 training, batch 4096, frames streamed "
                            f"from {n_files} PCM16 wav files x {secs:.0f} s through a {stream.capacity * 2 / 1e6:.1f} MB "
                            "ingest ring (smaller than the corpus), end to end from disk",
                "value": fps, "unit": "frames/s", "ms_per_step": ms / 40, "block_ms": [round(v, 3) for v in blocks],
                "h2d_bytes_per_step": uploaded / (7 * 40), "graph_stats_in_timed_region": d,
                "ingest": dict(stream.stats),
                "frac_of_bf16_sustained_peak": fps * FLOP_PER_FRAME / 1e12 / peaks["bf16_sustained"]}


def _stream_step(step_fn, pairs):
    cur, nxt = next(pairs)
    return step_fn(cur, next_data=nxt)


def leg_widened_inference(dev, peaks):
    """BASELINE.json configs[4]: widened VAE (segment_length 4096, n_units 4096, latent 256) inference over 1 M frames
    at hop 512, batches of 16 384: PCM16 wav in HBM -> frames -> encode -> reparameterize -> decode -> overlap-add
    across batch boundaries (inference.reconstruct_audio)."""
    from rawaudiovae_kelsey_b200 import inference as inf
    from rawvae.model import VAE
    Sw, Hw, Lw, hop, Bw, N = 4096, 4096, 256, 512, 16384, 1 << 20
    flop_per_frame = 73400320                    # SURVEY.md 8(a) a13
    torch.manual_seed(0)
    model = VAE(Sw, Hw, Lw).to(dev).eval()
    model.eps_seed = 3
    n_samples = (N - 1) * hop + Sw
    wav = torch.randint(-20000, 20000, (n_samples,), dtype=torch.int16, device=dev)
    inf.reconstruct_audio(model, wav[:(4 * Bw - 1) * hop + Sw], hop=hop, batch_size=Bw)       # warm-up: plans, tensor maps
    torch.cuda.synchronize()
    times = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = inf.reconstruct_audio(model, wav, hop=hop, batch_size=Bw)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    assert out.numel() == n_samples and bool(torch.isfinite(out[::4097]).all())
    ms = float(np.median(times))
    fps = N / (ms * 1e-3)
    tf = fps * flop_per_frame / 1e12
    return {"workload": "widened VAE (S=4096,H=4096,L=256) bf16 inference, 1 Mi frames at hop 512, batch 16384: "
                        "frames -> encode -> reparameterize -> decode -> overlap-add",
            "value": fps, "unit": "frames/s", "ms_total": ms, "runs_ms": [round(v, 2) for v in times],
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                         "frac": tf / peaks["bf16_sustained"], "frac_of_burst": tf / peaks["bf16_burst"],
                         "peak_kind": f"bf16_tflops_sustained ({peaks['source']}): ~{ms:.0f} ms of back-to-back GEMMs"}}


def extra_legs(dev, audio, n_frames, peaks):
    out = {}
    for name, fn in (("fp32_mode", lambda: leg_fp32_mode(dev, audio, n_frames, peaks)),
                     ("stream_4096", lambda: leg_stream_4096(dev, peaks)),
                     ("widened_inference", lambda: leg_widened_inference(dev, peaks))):
        try:
            out[name] = fn()
        except Exception as e:   # a failing side leg must never take the headline line down
            out[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--files", type=int, default=32)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sustained", action=argparse.BooleanOptionalAction, default=False,
                    help="continue each leg for ~0.4 s of later blocks after the timed steps (key `sustained`)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the side legs (fp32 mode, kelsey_iterable.ini streaming, widened-VAE inference)")
    ap.add_argument("--blocks", type=int, default=1,
                    help="timed blocks of --steps steps each per leg (median reported)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="enqueue every step eagerly (no CUDA graph)")
    ap.add_argument("--no-prefetch", dest="prefetch", action="store_false",
                    help="every step gathers its own batch (no background prefetch of the next one)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU arm's step (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the product path has no CPU fallback"}))
        return 1
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
