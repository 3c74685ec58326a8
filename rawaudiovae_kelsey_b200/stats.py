"""TensorBoard parameter histograms computed on the GPU.

The reference logs `writer.add_histogram(name, param, step)` for every parameter (train_iterable.py:216-217 per batch,
train.py:203-204 per epoch). Each such call synchronises the device, copies the parameter to the host and sorts it
with np.histogram. `ParamHistogramLogger` instead bins all parameters in one kernel launch (rvae_param_histogram)
against TensorBoard's default bins and brings back only the bucket counts and moments, asynchronously; the host then
only writes the events. The events are those of add_histogram, except for the last bits of `sum` and `sum_squares`
(fp64, summed in a fixed order on the device rather than in numpy's order).
"""
from __future__ import annotations

import time
from collections import deque
from typing import List, Tuple

import numpy as np
import torch

from . import ops


def default_bins() -> List[float]:
    """SummaryWriter.default_bins (the bins of add_histogram(bins="tensorflow")): the same loop, so the same floats."""
    v = 1e-12
    buckets, neg_buckets = [], []
    while v < 1e20:
        buckets.append(v)
        neg_buckets.append(-v)
        v *= 1.1
    return neg_buckets[::-1] + [0] + buckets


def trim_histogram(counts: np.ndarray, edges: np.ndarray) -> Tuple[List[float], List[int]]:
    """(bucket_limit, bucket) of make_histogram for the full per-bin counts: the support of the histogram plus one
    empty leading bucket, with the matching right bin limits. Raises ValueError for an empty histogram, as
    make_histogram does."""
    cum_counts = np.cumsum(np.greater(counts, 0))
    start, end = np.searchsorted(cum_counts, [0, cum_counts[-1] - 1], side="right")
    start, end = int(start), int(end) + 1
    counts = counts[start - 1:end] if start > 0 else np.concatenate([[0], counts[:end]])
    limits = np.asarray(edges)[start:end + 1]
    if counts.size == 0 or limits.size == 0:
        raise ValueError("The histogram is empty, please file a bug report.")
    return limits.tolist(), [int(c) for c in counts]


def histogram_fields(counts, edges, vmin, vmax, num, vsum, sum_squares) -> dict:
    """Keyword arguments of SummaryWriter.add_histogram_raw for one parameter's record fields."""
    limits, buckets = trim_histogram(np.asarray(counts), edges)
    return {"min": float(vmin), "max": float(vmax), "num": int(num), "sum": float(vsum),
            "sum_squares": float(sum_squares), "bucket_limits": limits, "bucket_counts": buckets}


class ParamHistogramLogger:
    """Histograms of every parameter of a VAE, written with `writer.add_histogram_raw` under the parameter names.

        hist = ParamHistogramLogger(model, writer)
        hist.record(step)          # after the step's call returned, on the same stream: never synchronises
        ...
        hist.flush()               # write the records whose copies have completed
        hist.flush(wait=True)      # write all of them (checkpoints, end of run)

    `record` launches the histogram kernel on the current stream over the model's flat parameter buffer, so it sees
    the parameters exactly as the work enqueued before it left them, and copies the record into a pinned host slot
    of a small ring. When every slot is taken it first writes the oldest one, waiting only for that slot's copy."""

    def __init__(self, model, writer, slots: int = 4):
        self.model, self.writer = model, writer
        self.names = [n for n, _ in model.named_parameters()]
        self.edges = np.asarray(default_bins(), dtype=np.float64)
        self.layout = ops.histogram_record_layout(len(self.names), self.edges.size)
        nbytes = self.layout["bytes"]
        self._host = [torch.empty(nbytes, dtype=torch.uint8, pin_memory=True) for _ in range(max(1, int(slots)))]
        self._events = [torch.cuda.Event() for _ in self._host]
        self._free = list(range(len(self._host)))
        self._pending = deque()   # (slot, step, walltime) in record order
        self._dev = None
        self._segs = None         # (flat buffer, offsets, lengths) of the last record

    def _segments(self):
        flat = self.model._ensure_flat()
        if self._segs is None or self._segs[0] is not flat.params:
            # each parameter as rows of its padded block (one row when contiguous): the padding is not counted
            offs, rows, cols, pitch = [], [], [], []
            for n in self.names:
                off, shape, strides = flat.geometry[n]
                offs.append(off)
                if len(shape) == 2 and strides[0] != shape[1]:
                    rows.append(shape[0]); cols.append(shape[1]); pitch.append(strides[0])
                else:
                    n_el = int(np.prod(shape))
                    rows.append(1); cols.append(n_el); pitch.append(n_el)
            a = lambda v: np.asarray(v, np.int64)
            self._segs = (flat.params, a(offs), a(rows), a(cols), a(pitch))
        return self._segs

    def record(self, step: int) -> None:
        params, offs, rows, cols, pitch = self._segments()
        if not self._free:
            self._write(self._pending.popleft())
        slot = self._free.pop()
        if self._dev is None or self._dev.device != params.device:
            self._dev = torch.empty(self.layout["total"], dtype=torch.uint8, device=params.device)
        if (rows == 1).all():
            ops.param_histogram(params, offs, cols, self.edges, out=self._dev)
        else:
            ops.param_histogram(params, offs, cols, self.edges, out=self._dev, seg_rows=rows, seg_pitch=pitch)
        self._host[slot].copy_(self._dev[:self.layout["bytes"]], non_blocking=True)
        self._events[slot].record()
        self._pending.append((slot, int(step), time.time()))

    def flush(self, wait: bool = False) -> None:
        """Write every record whose copy has completed (wait=True: every record)."""
        while self._pending:
            if not wait and not self._events[self._pending[0][0]].query():
                break
            self._write(self._pending.popleft())

    def _write(self, item) -> None:
        slot, step, walltime = item
        self._events[slot].synchronize()
        r = ops.unpack_histogram_record(self._host[slot], len(self.names), self.edges.size)
        try:
            for i, name in enumerate(self.names):
                self.writer.add_histogram_raw(name, **histogram_fields(
                    r["counts"][i], self.edges, r["min"][i], r["max"][i], r["num"][i], r["sum"][i],
                    r["sum_squares"][i]), global_step=step, walltime=walltime)
        finally:
            self._free.append(slot)
