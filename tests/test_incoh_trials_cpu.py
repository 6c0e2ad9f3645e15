"""Host logic of pb.incoherent_dedispersion_trials: the delay table and the rows shared by every
trial DM (incoherent_trial_delays) against the oracle's incoherent dedispersion per DM, and the
refusals that come before any device work.  No GPU needed."""

import numpy as np
import pytest

import pulsarbat_b200 as pb
from oracle import pbk_oracle as orc
from pulsarbat_b200.transforms.dedispersion import incoherent_trial_delays

u = pb.units
SR, FCEN, BW = 1e3, 600e6, 10e6


def _signal(n=4096, nchan=8, data=None, dtype=np.float32, freq_align="center"):
    x = np.zeros((n, nchan), dtype) if data is None else data
    return pb.IntensitySignal(x, sample_rate=SR * u.Hz, center_freq=FCEN * u.Hz,
                              chan_bw=BW * u.Hz, freq_align=freq_align)


@pytest.mark.parametrize("dms", [(30.0,), (30.0, 12.0), (0.0,), (12.0, 0.0, -8.0, 12.0),
                                 (-20.0, -3.0), (5.0, 5.0, 5.0), (40.0, -40.0, 0.5)])
@pytest.mark.parametrize("ref", ["center", "top", "bottom"])
@pytest.mark.parametrize("nchan,align", [(8, "center"), (7, "center"), (16, "top"), (1, "center")])
def test_delays_match_the_oracle_per_dm(dms, ref, nchan, align):
    rng = np.random.default_rng(11)
    n = 4096
    x = rng.integers(0, 16, size=(n, nchan)).astype(np.float32)
    z = _signal(n=n, nchan=nchan, data=x, freq_align=align)
    rf = {"center": z.center_freq, "top": z.max_freq, "bottom": z.min_freq}[ref]
    e, t_lo, rows = incoherent_trial_delays(z, [pb.DM(d) for d in dms], rf)
    assert e.shape == (len(dms), nchan) and e.dtype == np.int64
    valid = []
    for k, dm in enumerate(dms):
        y, cb, delays = orc.incoherent_dedispersion(x, dm, sample_rate=SR, center_freq=FCEN,
                                                    chan_bw=BW, freq_align=z.freq_align,
                                                    ref_freq=float(u.to_value(rf, u.Hz)))
        # the table is the oracle's delays less its crop, moved to the first shared row
        assert np.array_equal(e[k], delays - cb + t_lo)
        valid.append((cb, cb + len(y)))
        # every shared row is a valid row of this trial, and its sum is the oracle's row sum
        assert cb <= t_lo and t_lo + rows <= cb + len(y)
        want = y[t_lo - cb:t_lo - cb + rows].astype(np.int64).sum(axis=1)
        got = np.stack([x[t_lo + j + delays - cb, np.arange(nchan)] for j in range(rows)]
                       ).astype(np.int64).sum(axis=1) if rows else np.zeros(0, np.int64)
        assert np.array_equal(got, want)
    assert t_lo == max(v[0] for v in valid)
    assert rows == max(0, min(v[1] for v in valid) - t_lo)
    assert e.min() >= 0 and (rows == 0 or e.max() + rows <= n)


def test_empty_intersection_gives_zero_rows():
    z = _signal(n=512)
    # each sweep alone fits the signal, but their valid rows sit at opposite ends of it
    dms = [pb.DM(120.0), pb.DM(-120.0)]
    for d in dms:
        _, n_out, _ = pb.transforms.dedispersion.incoherent_delays(z, d, z.max_freq)
        assert n_out > 0
    _, _, rows = incoherent_trial_delays(z, dms, z.max_freq)
    assert rows == 0


def test_refusals():
    z = _signal()
    with pytest.raises(TypeError, match="RadioSignal"):
        pb.incoherent_dedispersion_trials(np.zeros((64, 4), np.float32), [1.0])
    with pytest.raises(TypeError, match="RadioSignal"):
        pb.incoherent_dedispersion_trials(pb.Signal(np.zeros((64, 4), np.float32),
                                                    sample_rate=SR * u.Hz), [1.0])
    with pytest.raises(TypeError, match="float32"):
        pb.incoherent_dedispersion_trials(_signal(dtype=np.float64), [1.0])
    zc = pb.BasebandSignal(np.zeros((64, 4), np.complex64), sample_rate=SR * u.Hz,
                           center_freq=FCEN * u.Hz)
    with pytest.raises(TypeError, match="float32"):
        pb.incoherent_dedispersion_trials(zc, [1.0])
    with pytest.raises(ValueError, match="sweep exceeds"):
        pb.incoherent_dedispersion_trials(z, [1.0, 5000.0])
    with pytest.raises(ValueError, match="sweep exceeds"):
        incoherent_trial_delays(z, [5000.0], z.center_freq)
    with pytest.raises(ValueError):
        pb.incoherent_dedispersion_trials(z, [])
    with pytest.raises(TypeError):
        pb.incoherent_dedispersion_trials(z, 3.0)


def test_sweep_error_is_the_one_of_incoherent_dedispersion():
    z = _signal(n=256)
    with pytest.raises(ValueError) as single:
        pb.incoherent_dedispersion(z, pb.DM(500.0))
    with pytest.raises(ValueError) as many:
        pb.incoherent_dedispersion_trials(z, [0.0, 500.0])
    assert str(single.value) == str(many.value)


def test_dask_input_raises(monkeypatch):
    import fake_dask
    da = fake_dask.install(monkeypatch)
    z = _signal(data=da.from_array(np.zeros((4096, 8), np.float32), chunks=(4096, 4)))
    with pytest.raises(TypeError, match="incoherent_dedispersion per chunk"):
        pb.incoherent_dedispersion_trials(z, [1.0, 2.0])
