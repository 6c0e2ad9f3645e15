"""Host side of the single-pulse search: the float64 definition (tests/single_pulse_oracle.py)
against brute-force loops, window partitioning, the defaults and refusals of
pb.single_pulse_search, and its choice between passing the trials' array by view and stacking.
No GPU needed."""

import itertools
import math

import numpy as np
import pytest

import pulsarbat_b200 as pb
import single_pulse_oracle as spo
from pulsarbat_b200.pulsar import search

u = pb.units


def brute(x, widths, window):
    """Every (t, w) in plain Python loops, from the definition."""
    nser, rows, ncols = x.shape
    nwin = -(-rows // window)
    snr = np.full((nser, nwin, ncols), -np.inf)
    start = np.full((nser, nwin, ncols), -1)
    width = np.full((nser, nwin, ncols), -1)
    for s, c in itertools.product(range(nser), range(ncols)):
        col = [float(v) for v in x[s, :, c]]
        mean = sum(col) / rows
        std = math.sqrt(sum((v - mean) ** 2 for v in col) / rows)
        for j in range(nwin):
            best = None
            for t in range(j * window, min((j + 1) * window, rows)):
                for w in widths:
                    if t + w > rows:
                        continue
                    v = (sum(col[t:t + w]) - w * mean) / (std * math.sqrt(w)) if std > 0 else 0.0
                    if best is None or v > best[0]:    # scanning t then w ascending: first max
                        best = (v, t, w)
            if best is not None:
                snr[s, j, c], start[s, j, c], width[s, j, c] = best
    return snr, start, width


@pytest.mark.parametrize("rows,ncols,widths,window", [
    (37, 1, (1,), 1), (37, 2, (1, 3, 4), 5), (40, 3, (2, 5, 16), 7), (23, 1, (1, 2, 4, 8), 23),
    (23, 2, (3, 30), 4), (16, 1, (1, 2, 4), 100), (9, 2, (10, 12), 3)])
def test_oracle_matches_brute_force(rows, ncols, widths, window):
    rng = np.random.default_rng(rows * 7 + ncols)
    x = rng.integers(0, 6, size=(2, rows, ncols)).astype(np.float32)
    x[1, :, 0] = 3.0                                      # std = 0: every S/N is 0
    want = brute(x, widths, window)
    got = spo.boxcar_search(x, widths, window)
    assert np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2])
    assert np.allclose(got[0], want[0], rtol=1e-12, atol=1e-12)
    st = spo.series_stats(x)
    assert st.shape == (2, ncols, 2)
    assert np.allclose(st[..., 0], x.astype(np.float64).mean(1), rtol=1e-15, atol=0)


def test_window_partitioning():
    x = np.random.default_rng(1).standard_normal((1, 10, 1)).astype(np.float32)
    # a partial last window: 10 starts in windows of 4 -> 4, 4, 2
    snr, start, width = spo.boxcar_search(x, (1, 2), 4)
    assert snr.shape == (1, 3, 1)
    assert list(start[0, :, 0] // 4) == [0, 1, 2]
    # window > rows: one window; widths > rows: no valid pair
    snr, start, width = spo.boxcar_search(x, (1,), 50)
    assert snr.shape == (1, 1, 1) and 0 <= start[0, 0, 0] < 10
    snr, start, width = spo.boxcar_search(x, (11, 20), 3)
    assert snr.shape == (1, 4, 1)
    assert np.all(snr == -np.inf) and np.all(start == -1) and np.all(width == -1)
    # the last start of a width is rows - w: its window still sees it
    snr, start, width = spo.boxcar_search(x, (10,), 3)
    assert list(start[0, :, 0]) == [0, -1, -1, -1] and list(width[0, :, 0]) == [10, -1, -1, -1]


def _trials(n=3, rows=64, ncols=1, data=None, dtype=np.float32):
    x = np.zeros((n, rows, ncols), dtype) if data is None else data
    return [pb.IntensitySignal(x[k], sample_rate=1e3 * u.Hz, center_freq=600e6 * u.Hz,
                               chan_bw=1e6 * u.Hz, start_time=pb.Time(59000.0, format="mjd"))
            for k in range(n)]


def test_defaults():
    import inspect
    sig = inspect.signature(pb.single_pulse_search)
    assert sig.parameters["threshold"].default == 6.0
    assert search.DEFAULT_WIDTHS == tuple(2 ** k for k in range(11))
    assert "single_pulse_search" in pb.pulsar.__all__ and pb.single_pulse_search is \
        search.single_pulse_search


def test_refusals():
    with pytest.raises(ValueError):
        pb.single_pulse_search([])
    with pytest.raises(TypeError, match="IntensitySignal"):
        pb.single_pulse_search([np.zeros((8, 1), np.float32)])
    with pytest.raises(TypeError, match="float32"):
        pb.single_pulse_search(_trials(dtype=np.float64))
    t = _trials()
    other = _trials(rows=32)[0]
    with pytest.raises(ValueError, match="shape"):
        pb.single_pulse_search(t + [other])
    slow = pb.IntensitySignal(np.zeros((64, 1), np.float32), sample_rate=2e3 * u.Hz,
                              center_freq=600e6 * u.Hz, chan_bw=1e6 * u.Hz,
                              start_time=pb.Time(59000.0, format="mjd"))
    with pytest.raises(ValueError, match="sample rate"):
        pb.single_pulse_search(t + [slow])
    late = pb.IntensitySignal(np.zeros((64, 1), np.float32), sample_rate=1e3 * u.Hz,
                              center_freq=600e6 * u.Hz, chan_bw=1e6 * u.Hz,
                              start_time=pb.Time(59001.0, format="mjd"))
    with pytest.raises(ValueError, match="start time"):
        pb.single_pulse_search(t + [late])


def test_dask_input_raises(monkeypatch):
    import fake_dask
    da = fake_dask.install(monkeypatch)
    z = pb.IntensitySignal(da.from_array(np.zeros((64, 1), np.float32), chunks=(32, 1)),
                           sample_rate=1e3 * u.Hz, center_freq=600e6 * u.Hz, chan_bw=1e6 * u.Hz)
    with pytest.raises(TypeError, match="dask"):
        pb.single_pulse_search([z])


def test_view_or_stack(monkeypatch):
    x = np.arange(3 * 64 * 2, dtype=np.float32).reshape(3, 64, 2)
    datas = [x[k] for k in range(3)]

    def refuse(_):
        raise AssertionError("the trials are slabs of one array: no stack expected")
    monkeypatch.setattr(search, "_stack", refuse)
    plane = search._plane(datas)
    assert plane.shape == x.shape and np.shares_memory(plane, x)
    assert np.array_equal(plane, x)
    assert np.array_equal(search._plane(datas[:1]), x[:1])
    # out of order, separate arrays, or strided slabs are stacked
    calls = []
    monkeypatch.setattr(search, "_stack", lambda d: calls.append(len(d)) or np.stack(d))
    for ds in ([datas[1], datas[0]], [datas[0].copy(), datas[1].copy()],
               [x[:, :, 0][k] for k in range(2)], [datas[0], datas[2]]):
        plane = search._plane(ds)
        assert np.array_equal(plane, np.stack(ds))
    assert calls == [2, 2, 2, 2]
