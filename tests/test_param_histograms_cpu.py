"""Host side of the GPU parameter histograms (rawaudiovae_kelsey_b200.stats): the edge table, the trimming of the
full per-bin counts and the fields handed to SummaryWriter.add_histogram_raw, checked against TensorBoard's own
make_histogram / histogram(). The counts fed in here are np.histogram's, i.e. what the kernel must produce (checked
on the GPU in test_gpu_param_histograms.py)."""
import numpy as np
import pytest

pytest.importorskip("tensorboard")
from torch.utils.tensorboard import SummaryWriter  # noqa: E402
from torch.utils.tensorboard.summary import histogram, histogram_raw, make_histogram  # noqa: E402

from rawaudiovae_kelsey_b200 import stats  # noqa: E402

EDGES = np.asarray(stats.default_bins(), dtype=np.float64)


def test_edge_table_equals_summary_writer_default_bins(tmp_path):
    w = SummaryWriter(log_dir=str(tmp_path))
    try:
        ref = np.asarray(w.default_bins, dtype=np.float64)
    finally:
        w.close()
    assert EDGES.shape == ref.shape == (1549,)
    assert EDGES.tobytes() == ref.tobytes()
    assert np.all(np.diff(EDGES) > 0)


def _cases():
    rng = np.random.default_rng(0)
    e = EDGES
    return {
        "uniform_init": rng.uniform(-0.03, 0.03, 5000).astype(np.float32),
        "normal": rng.normal(0, 1.0, 3000).astype(np.float32),
        "all_zero": np.zeros(2048, np.float32),
        "single_bin": np.full(100, 0.0237, np.float32),
        "first_bin": np.array([e[0], e[0] * 0.9999999, e[0]], np.float64),
        "last_bin": np.array([e[-1], e[-2] * 1.0000001, e[-1]], np.float64),
        "both_ends": np.array([e[0], 0.5, e[-1]], np.float64),
        "outside_and_nan": np.array([np.nan, np.inf, -np.inf, 3.4e38, -3.4e38, 1.0, -2.0], np.float64),
    }


@pytest.mark.parametrize("name", list(_cases()))
def test_trim_matches_make_histogram(name):
    values = _cases()[name].astype(np.float64)
    ref = make_histogram(values, EDGES)
    counts, _ = np.histogram(values, bins=EDGES)
    limits, buckets = stats.trim_histogram(counts.astype(np.int32), EDGES)
    assert limits == list(ref.bucket_limit)
    assert buckets == list(ref.bucket)


def test_trim_of_an_empty_histogram_raises_like_make_histogram():
    with pytest.raises(ValueError):
        make_histogram(np.array([np.nan, np.inf]), EDGES)
    with pytest.raises(ValueError):
        stats.trim_histogram(np.zeros(1548, np.int32), EDGES)


@pytest.mark.parametrize("name", list(_cases()))
def test_raw_fields_serialise_like_histogram(name):
    values = _cases()[name]
    v64 = values.astype(np.float64)
    counts, _ = np.histogram(v64, bins=EDGES)
    f = stats.histogram_fields(counts.astype(np.int32), EDGES, v64.min(), v64.max(), v64.size, v64.sum() + 1.0,
                               v64.dot(v64) * 2.0)
    ref = histogram("p", values, EDGES)
    got = histogram_raw("p", f["min"], f["max"], f["num"], f["sum"], f["sum_squares"], f["bucket_limits"],
                        f["bucket_counts"])
    got.value[0].histo.sum = ref.value[0].histo.sum
    got.value[0].histo.sum_squares = ref.value[0].histo.sum_squares
    assert got.SerializeToString() == ref.SerializeToString()
