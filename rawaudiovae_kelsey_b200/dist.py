"""Batch-sharded data parallelism: one process per GPU, torch.distributed (NCCL over NVLink / NVSwitch) as plumbing.

The reference has no distributed code (SURVEY.md 2b); this is the new subsystem (5) of the north star. Frames are
independent units, so the path shards with exactly one exchange step per optimizer step:

  * every rank holds the full model + Adam state (23 MB + 46 MB) and the wav corpus; rank r takes rows
    shard_bounds(B, r, W) of each global batch (dataset.GpuFrameLoader / GpuFrameStream);
  * the loss is normalised by the GLOBAL batch size inside the epilogues (rvae_plan_set_global_batch), so a plain
    SUM all-reduce of the gradients equals the single-process gradient of the concatenated batch exactly - also
    for unequal shards;
  * gradients are all-reduced in 5 buckets in backward-completion order (W4, W3, W2 + biases, W1) by NCCL calls the
    C library issues itself (rvae_plan_train_step, include/rvae_b200.h "Data parallelism"): each runs on a
    communication stream right after the backward stage that completes it, on the SMs the persistent GEMM grids leave
    free, while the remaining dgrad / wgrad GEMMs run; each bucket's Adam launch waits for its reduced gradient.
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch
import torch.distributed as dist

from .model import _StepBase


def init_from_env(backend: Optional[str] = None) -> tuple:
    """Initialise torch.distributed from torchrun's environment. Returns (rank, world, local_rank)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
            dist.init_process_group(backend, rank=rank, world_size=world,
                                    device_id=torch.device("cuda", local_rank))
        else:
            dist.init_process_group(backend, rank=rank, world_size=world)
    return rank, world, local_rank


def allreduce_buckets(buckets: List[torch.Tensor], group=None, async_op: bool = True) -> list:
    """SUM all-reduce each bucket in order; returns the work handles (call .wait() before consuming)."""
    works = []
    for b in buckets:
        w = dist.all_reduce(b, op=dist.ReduceOp.SUM, group=group, async_op=async_op)
        if async_op:
            works.append(w)
    return works


def broadcast_parameters(flat_params: torch.Tensor, group=None, src: int = 0) -> None:
    """Make every replica start from rank `src`'s weights."""
    dist.broadcast(flat_params, src=src, group=group)


def _libnccl_path() -> Optional[str]:
    """The libnccl.so.2 torch itself uses (nvidia-nccl wheel), so both share one NCCL in the process."""
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for loc in (spec.submodule_search_locations or []):
            cand = os.path.join(loc, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                return cand
    except Exception:
        pass
    return None


_COMM_READY = set()
_SYM_READY = {}


class _DevBuffer:
    """A raw device allocation exposed through __cuda_array_interface__ (so torch can view it without copying)."""

    def __init__(self, ptr: int, n_float32: int):
        self.__cuda_array_interface__ = {"shape": (n_float32,), "typestr": "<f4", "data": (ptr, False), "version": 3}


_SYMM_KEEP = []   # (buffer tensor, rendezvous handle): the symmetric allocations stay alive with the process


def _adopt_torch_symmetric(lib, flat, group, rank, world):
    """Gradient buffer [flag area | total fp32] in torch symmetric memory, mapped by every rank, with its NVLS multicast
    mapping handed to the library (rvae_dp_sym_adopt). Returns the gradient tensor, or None when ANY rank could not
    set it up (then nobody uses it)."""
    from . import _lib, ops
    import ctypes as C
    ok, buf, hdl, err = True, None, None, ""
    flag_bytes = int(lib.rvae_dp_sym_flag_bytes())
    n_data = (flat.total + 63) // 64 * 64
    try:
        import torch.distributed._symmetric_memory as symm_mem
        g = group if group is not None else dist.group.WORLD
        with torch.cuda.device(flat.device):
            buf = symm_mem.empty(flag_bytes // 4 + n_data, dtype=torch.float32, device=flat.device)
            buf.zero_()
            torch.cuda.synchronize(flat.device)
            hdl = symm_mem.rendezvous(buf, g)
        off = buf.data_ptr() - int(hdl.buffer_ptrs[rank])
        ok = off >= 0 and len(hdl.buffer_ptrs) == world and (buf.data_ptr() % 256) == 0
    except Exception as e:   # no symmetric memory on this build / box: fall back, on every rank
        ok, err = False, repr(e)[:200]
    box = [None] * world
    dist.all_gather_object(box, ok, group=group)
    if not all(box):
        if not ok and rank == 0:
            print(f"[rank {rank}] torch symmetric memory unavailable ({err}); using the CUDA-IPC gradient buffer", flush=True)
        return None
    peers = (C.c_void_p * world)(*[int(hdl.buffer_ptrs[p]) + off for p in range(world)])
    mc = int(hdl.multicast_ptr) + off if int(hdl.multicast_ptr) else 0
    try:
        with torch.cuda.device(flat.device):
            _lib.check(lib.rvae_dp_sym_adopt(ops.ctx(flat.device), peers, C.c_void_p(mc or None), n_data * 4, rank, world))
    except _lib.RvaeError as e:
        ok = False
        print(f"[rank {rank}] rvae_dp_sym_adopt failed ({e})", flush=True)
    box = [None] * world
    dist.all_gather_object(box, ok, group=group)
    if not all(box):
        raise RuntimeError("data parallel set-up: rvae_dp_sym_adopt failed on some ranks (see above)")
    _SYMM_KEEP.append((buf, hdl))
    dist.barrier(group=group)      # every rank's flag area is zeroed and mapped before anyone signals
    return buf[flag_bytes // 4: flag_bytes // 4 + flat.total]


def _move_grads(model, flat, grads):
    if flat.grads.data_ptr() != grads.data_ptr():
        grads.copy_(flat.grads)
        flat.grads = grads
        model._plans = {}              # plans bind raw pointers: rebuild them on the new gradient buffer
        for _, p in model._named():
            p.grad = None


def adopt_symmetric_grads(model, group=None, peer_loads: bool = False) -> bool:
    """Move the model's flat gradient buffer into a symmetric allocation that every rank of the group maps over
    CUDA IPC, so the gradient all-reduce can be done by librvae_b200's own NVLink peer-memory kernel instead of NCCL.
    Returns False (and leaves NCCL in charge) when RVAE_DP_BACKEND=nccl or the group has more than 8 ranks.
    peer_loads=True (deterministic steps): the peer-load exchange, which sums the ranks in rank order, whatever
    RVAE_DP_BACKEND says; raises ValueError naming the backend when the group ends up on NVLS multicast or NCCL."""
    from . import _lib, ops
    if peer_loads:
        if dist.get_world_size(group) > 8:     # (no GPU work yet: the peer-load kernel takes at most 8 ranks)
            agree_peer_loads("nccl", group)
        flat = model._ensure_flat()
        ok = _adopt(model, group, "p2p")
        agree_peer_loads(("nvls" if _lib.load().rvae_dp_uses_multicast(ops.ctx(flat.device)) else "p2p") if ok
                         else "nccl", group)
        return True
    return _adopt(model, group, os.environ.get("RVAE_DP_BACKEND", "auto"))


def agree_peer_loads(backend: str, group=None) -> None:
    """Deterministic data parallelism: every rank passes the exchange its gradients ended up on ("p2p" = peer loads,
    "nvls", "nccl"); all ranks raise ValueError naming the other backends unless every rank is on peer loads, so no
    rank trains on while another refuses, and none trains non-deterministically."""
    box = [None] * dist.get_world_size(group)
    dist.all_gather_object(box, backend, group=group)
    bad = sorted({b for b in box if b != "p2p"})
    if bad:
        raise ValueError(f"deterministic data parallelism needs the peer-load gradient all-reduce (ranks summed in "
                         f"rank order); this group exchanges gradients by {' / '.join(bad)}, which gives no order "
                         f"guarantee")


def _adopt(model, group, backend) -> bool:
    from . import _lib, ops
    import ctypes as C
    flat = model._ensure_flat()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if backend == "nccl" or world > 8:
        return False
    key = flat.device.index
    if key in _SYM_READY:
        if _SYM_READY[key][1] != flat.total:
            return False               # one symmetric gradient buffer per device: other models use NCCL
        grads = _SYM_READY[key][0]
    else:
        lib = _lib.load()
        # First choice: a symmetric allocation from torch.distributed's symmetric memory (plumbing: it creates, exchanges
        # and maps the handles) WITH an NVLS multicast mapping, so the all-reduce kernel reduces in the NVSwitch.
        # Default ("auto"): from 3 ranks up. Measured on one box (profiles/README.md): N = 8 +5.4 %, N = 4 +2.6 %, N = 2
        # -3.5 % (with two ranks a rank's own slice travels to the switch and back for nothing), so two ranks keep the
        # library's own CUDA-IPC allocation and peer loads. RVAE_DP_BACKEND=nvls / p2p / nccl force one.
        if backend == "nvls" or (backend == "auto" and world >= 3):
            grads = _adopt_torch_symmetric(lib, flat, group, rank, world)
            if grads is not None:
                _SYM_READY[key] = (grads, flat.total)
                _move_grads(model, flat, grads)
                return True
        # Every step below is agreed on by ALL ranks before anyone relies on it: if a single rank cannot allocate,
        # export or map the buffers (no CUDA IPC in this container, no peer access), the whole group stays on NCCL.
        ptr, handle = C.c_void_p(), (C.c_char * 64)()
        ok = True
        with torch.cuda.device(flat.device):
            try:
                _lib.check(lib.rvae_dp_sym_alloc(ops.ctx(flat.device), flat.total * 4, C.byref(ptr), handle))
            except _lib.RvaeError as e:
                ok = False
                print(f"[rank {rank}] symmetric gradient buffer unavailable ({e}); using NCCL", flush=True)
            box = [None] * world
            dist.all_gather_object(box, (ok, bytes(handle)), group=group)
            if not all(o for o, _ in box):
                _SYM_READY[key] = (None, -1)
                return False
            try:
                _lib.check(lib.rvae_dp_sym_open(ops.ctx(flat.device), b"".join(h for _, h in box), rank, world))
            except _lib.RvaeError as e:
                ok = False
                print(f"[rank {rank}] cannot map the peers' gradient buffers ({e}); using NCCL", flush=True)
            box = [None] * world
            dist.all_gather_object(box, ok, group=group)
            if not all(box):
                _SYM_READY[key] = (None, -1)
                return False
        grads = torch.as_tensor(_DevBuffer(ptr.value, flat.total), device=flat.device)
        _SYM_READY[key] = (grads, flat.total)
    if flat.grads.data_ptr() != grads.data_ptr():
        grads.copy_(flat.grads)
        flat.grads = grads
        model._plans = {}              # plans bind raw pointers: rebuild them on the new gradient buffer
        for _, p in model._named():
            p.grad = None
    return True


def check_health(device: Optional[torch.device] = None) -> None:
    """Raise if the peer-memory all-reduce recorded a barrier timeout (a rank that stopped taking part). Reads 4
    bytes synchronously: call it where the host synchronises anyway (loss read-back, checkpoints)."""
    from . import _lib, ops
    import ctypes as C
    st = C.c_uint(0)
    _lib.check(_lib.load().rvae_dp_status(ops.ctx(device), C.byref(st)))
    if st.value:
        v = st.value
        raise RuntimeError(f"data-parallel all-reduce timed out waiting for rank {(v >> 8) & 0xff} "
                           f"(flag set {(v >> 4) & 0xf}, phase {v & 0xf}); gradients since then are invalid")


def sync_ranks(group=None) -> None:
    """Host-level barrier (no-op in a single process). The trainers call it after every rank-0-only block
    (checkpoints, histograms, test-audio reconstruction) so that no rank runs ahead into an all-reduce the others
    only join once rank 0 is back."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.barrier(group)


def agree(value, group=None, src: int = 0):
    """Every rank gets rank `src`'s value of a picklable object (sampler seeds, file orders)."""
    if not (dist.is_initialized() and dist.get_world_size(group) > 1):
        return value
    box = [value]
    dist.broadcast_object_list(box, src=src, group=group)
    return box[0]


def init_native_comm(device: torch.device, group=None) -> None:
    """Create librvae_b200's own NCCL communicator for `device`: rank 0 draws the 128-byte NCCL id, torch.distributed
    carries it to the other ranks (plumbing only), every rank calls rvae_dp_init. Idempotent."""
    from . import _lib, ops
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx in _COMM_READY:
        return
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    os.environ.setdefault("NCCL_MAX_CTAS", "16")   # the all-reduce kernels live on the SMs the GEMM grids leave free
    lib = _lib.load()
    path = _libnccl_path()
    cpath = path.encode() if path else None
    import ctypes as C
    buf = (C.c_char * 128)()
    if rank == 0:
        _lib.check(lib.rvae_dp_unique_id(ops.ctx(device), cpath, buf))
    box = [bytes(buf)]
    dist.broadcast_object_list(box, src=0, group=group)
    ident = (C.c_char * 128).from_buffer_copy(box[0])
    with torch.cuda.device(idx):
        _lib.check(lib.rvae_dp_init(ops.ctx(device), cpath, ident, rank, world))
    _COMM_READY.add(idx)


class DataParallelTrainStep(_StepBase):
    """FusedTrainStep for W ranks. The whole step, collectives included, is enqueued by ONE C call
    (rvae_plan_train_step): forward (+fused loss) -> backward stages, each followed by the NCCL all-reduce of the
    gradient bucket it completed on a communication stream, overlapped with the later stages -> Adam per bucket as its
    reduced gradient arrives. `data` is this rank's shard of the global batch; `next_data` (optional) the shard of
    the next call, prefetched in the background.

    The returned loss is the mean over THIS rank's frames (an unbiased estimate of the global mean that needs no
    collective); reduce_loss=True additionally averages it over the ranks (exact for equal shards).
    graph=True captures the whole step, NCCL collectives included, into one CUDA graph per input signature.
    schedule: as for FusedTrainStep; every rank evaluates it at the same step counter.
    max_grad_norm: as for FusedTrainStep. The norm is taken over the all-reduced gradient, which is identical on every
    rank, in a fixed order, so every rank clips by the same factor and the replicas stay bitwise equal.
    deterministic: as for FusedTrainStep, with the gradients exchanged by the peer-load all-reduce whatever
    RVAE_DP_BACKEND says (it sums the ranks in rank order). RVAE_DP_BACKEND=nvls or nccl raises ValueError here, and
    so does a group that cannot use peer loads, at its first step: the step never trains non-deterministically.
    ema: as for FusedTrainStep. Each rank updates its own average from the all-reduced update, which is identical on
    every rank, so the averages stay bitwise equal without any communication."""

    def __init__(self, model, optimizer, kl_beta: float, global_batch: Optional[int] = None, group=None,
                 ring: int = 64, reduce_loss: bool = False, graph: bool = False, schedule=None, max_grad_norm=None,
                 deterministic: bool = False, ema=None):
        super().__init__(model, optimizer, kl_beta, ring, graph, schedule=schedule, max_grad_norm=max_grad_norm,
                         deterministic=deterministic, ema=ema)
        forced = os.environ.get("RVAE_DP_BACKEND", "auto")
        if self.deterministic and forced in ("nvls", "nccl"):
            raise ValueError(f"deterministic=True needs the peer-load gradient all-reduce; RVAE_DP_BACKEND={forced} "
                             f"gives no order guarantee")
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.global_batch = global_batch
        self.reduce_loss = reduce_loss
        self._synced = False

    # Which rows of the global batch a shard holds. The sharding loaders (dataset.GpuFrameLoader / GpuFrameStream)
    # stamp it on the FrameBatch; otherwise equal contiguous shards of `global_batch` are assumed.
    def _rows(self, data):
        from .dataset import shard_bounds
        fb = data[0] if isinstance(data, (list, tuple)) and data else data
        n = sum(r.n_frames for r in data) if isinstance(data, (list, tuple)) else \
            (data.n_frames if hasattr(data, "n_frames") else data.numel() // self.model.segment_length)
        gb = getattr(fb, "global_batch", None)
        if gb is None:
            gb = self.global_batch if self.global_batch is not None else n * self.world
        row0 = getattr(fb, "global_row0", None)
        if row0 is None:
            row0 = shard_bounds(gb, self.rank, self.world)[0]
        return int(row0), int(gb)

    def _configure(self, plan, data):
        if self.world <= 1:
            plan.set_global_batch(0)
            return
        row0, gb = self._rows(data)
        plan.set_global_batch(gb)      # loss normalisation: the SUM over ranks is the gradient of the global batch
        plan.set_noise_rows(row0)      # Philox counters: the same seed on every rank draws disjoint rows of one tensor
        if not getattr(plan, "_dp_on", False):
            plan.enable_dp(True)
            plan._dp_on = True

    def _key_extra(self, data):
        return self._rows(data) if self.world > 1 else ()

    def _prefetch(self, plan, data, next_data, frame_idx, first_frame):
        if self.world > 1:             # the prefetched noise belongs to the NEXT batch's shard rows
            plan.set_noise_rows(self._rows(next_data)[0])
        super()._prefetch(plan, data, next_data, frame_idx, first_frame)
        if self.world > 1 and data is not None:
            plan.set_noise_rows(self._rows(data)[0])

    def _seed(self):
        return self._shared_seed if getattr(self, "_shared_seed", None) is not None else super()._seed()

    def _enqueue(self, plan):
        self._train_step(plan, zero_grads=True)

    def __call__(self, data, eps: Optional[torch.Tensor] = None, next_data=None) -> torch.Tensor:
        flat = self._prepare()
        if not self._synced and self.world > 1:
            init_native_comm(flat.device, self.group)
            adopt_symmetric_grads(self.model, self.group, peer_loads=self.deterministic)
            flat = self._prepare()
            broadcast_parameters(flat.params, self.group)
            flat.sync_shadow()
            # ONE noise stream for the whole group: rank 0's seed everywhere, decorrelated by global row (see _rows)
            box = [super()._seed()]
            dist.broadcast_object_list(box, src=0, group=self.group)
            self._shared_seed = int(box[0])
            self._synced = True
        slot = self._run(data, eps, next_data)
        self._calls = getattr(self, "_calls", 0) + 1
        if self.reduce_loss and self.world > 1:
            dist.all_reduce(slot, op=dist.ReduceOp.SUM, group=self.group)
            slot.div_(self.world)
        return slot
