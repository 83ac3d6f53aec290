"""CPU: the host side of the per-epoch error histograms -- hist_quantiles on hand-made counts, the header
constants, and toa_montecarlo's return value with and without a histogram (driven by a stand-in batch)."""
import re

import numpy as np
import pytest

from roskfpos_b200 import lib as L
from roskfpos_b200 import synth
from roskfpos_b200.batch import hist_quantiles


def test_header_constants():
    src = open(L.HEADER_PATH).read()
    got = {k: int(v) for k, v in re.findall(r"#define (KFPOS_HIST_\w+)\s+(\d+)", src)}
    assert got == {"KFPOS_HIST_ERR": L.HIST_ERR, "KFPOS_HIST_ERR_XY": L.HIST_ERR_XY, "KFPOS_HIST_NEES": L.HIST_NEES}


def test_hist_quantiles_brackets():
    edges = [1.0, 2.0, 3.0]
    counts = np.array([[0, 3, 1, 0],    # 3 values in [1, 2), 1 in [2, 3)
                       [0, 0, 0, 0],    # empty
                       [5, 0, 0, 5],    # half in the first bin, half in the last
                       [0, 0, 0, 2],    # all in the last bin
                       [1, 0, 0, 0]], dtype=np.uint64)
    lo, hi = hist_quantiles(counts, edges, [0.0, 0.5, 0.75, 0.95, 1.0])
    nan = np.nan
    exp_lo = [[1, 1, 1, 2, 2], [nan] * 5, [0, 0, 3, 3, 3], [3] * 5, [0] * 5]
    exp_hi = [[2, 2, 2, 3, 3], [nan] * 5, [1, 1, np.inf, np.inf, np.inf], [np.inf] * 5, [1] * 5]
    np.testing.assert_array_equal(lo, exp_lo)
    np.testing.assert_array_equal(hi, exp_hi)


def test_hist_quantiles_against_sorted_values():
    """The bracket holds the empirical quantile (the ceil(q n)-th smallest value) of the binned values."""
    rng = np.random.default_rng(7)
    edges = np.arange(1, 41) * 0.025
    vals = np.abs(rng.normal(0, 0.3, size=(20, 997)))
    counts = np.stack([np.bincount(np.searchsorted(edges, v, side="right"), minlength=41) for v in vals])
    qs = [0.01, 0.5, 0.95, 0.999]
    lo, hi = hist_quantiles(counts, edges, qs)
    for j, q in enumerate(qs):
        kth = np.sort(vals, axis=1)[:, max(1, int(np.ceil(q * 997))) - 1]
        assert ((lo[:, j] <= kth) & (kth < hi[:, j])).all()


def test_hist_quantiles_errors():
    with pytest.raises(ValueError):
        hist_quantiles(np.zeros((2, 3)), [1.0], [0.5])
    with pytest.raises(ValueError):
        hist_quantiles(np.zeros((2, 2)), [1.0], [1.5])


class FakeBatch:
    """Records the calls toa_montecarlo makes; returns deterministic rows."""
    model, N, device = L.MODEL_T6, 5, 0

    def __init__(self):
        self.calls, self.rows = [], 0

    def set_state(self, *a, **k):
        self.calls.append("set_state")

    def set_truth_traj(self, truth, stream=None):
        self.calls.append("set_truth_traj" if truth is not None else "unset_truth")
        self.rows = 0 if truth is None else len(truth)

    def replay_toa(self, *a, **k):
        self.calls.append("replay_toa")

    def epoch_stats(self, stream=None):
        return np.full((self.rows, 6), 1.0)

    def set_error_hist(self, edges, quantity="err"):
        self.calls.append("set_error_hist" if edges is not None else "unset_hist")
        self.bins = 0 if edges is None else len(edges) + 1

    def error_hist(self, stream=None):
        return np.ones((self.rows, self.bins), dtype=np.uint64)


@pytest.fixture
def fake_chunks(monkeypatch):
    def chunk(n_filters, epoch0, n, anchors, device, want_truth=False, want_x0=False, out=None, **kw):
        return dict(x0=np.zeros((6, n_filters)), truth=np.zeros((n, 3, n_filters)), ranges=None, dt=0.1)
    monkeypatch.setattr(synth, "toa_montecarlo_chunk", chunk)


def test_toa_montecarlo_default_return_unchanged(fake_chunks):
    b = FakeBatch()
    rows = synth.toa_montecarlo(b, 7, 3, synth.anchors_for(8))
    assert isinstance(rows, np.ndarray) and rows.shape == (7, 6)
    assert "set_error_hist" not in b.calls and "unset_hist" not in b.calls
    assert b.calls[-1] == "unset_truth"


def test_toa_montecarlo_with_hist(fake_chunks):
    b = FakeBatch()
    rows, counts = synth.toa_montecarlo(b, 7, 3, synth.anchors_for(8), hist=([0.1, 0.2], "err"))
    assert rows.shape == (7, 6) and counts.shape == (7, 3) and counts.dtype == np.uint64
    assert b.calls[0] == "set_error_hist" and b.calls[-2:] == ["unset_truth", "unset_hist"]
