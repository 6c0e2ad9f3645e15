"""Host logic of pb.dedisperse_trials: the crop shared by all trial DMs, DM argument
normalisation and the refusal of dask input.  No GPU needed."""

import numpy as np
import pytest

import pulsarbat_b200 as pb
from pulsarbat_b200.transforms.dedispersion import as_dm_list, common_crop_range, crop_range

SR, FCEN = 6.25e6, 625e6


def _signal(n=2 ** 16, nchan=8, data=None):
    x = np.zeros((n, nchan, 2), np.complex64) if data is None else data
    return pb.DualPolarizationSignal(x, sample_rate=SR * pb.units.Hz,
                                     center_freq=FCEN * pb.units.Hz, pol_type="linear")


@pytest.mark.parametrize("dms", [(3.0,), (3.0, 1.0, 2.5), (0.0,), (0.0, 0.0), (-2.0, -0.5),
                                 (-2.0, 0.0, 3.0), (1e-4, -1e-4)])
@pytest.mark.parametrize("ref", ["center", "top", "bottom"])
def test_common_crop_is_the_intersection_of_every_dm_crop(dms, ref):
    z = _signal()
    rf = {"center": z.center_freq, "top": z.max_freq, "bottom": z.min_freq}[ref]
    DMs = [pb.DM(d) for d in dms]
    start, stop = common_crop_range(z, DMs, rf)
    ranges = [crop_range(z, d, rf) for d in DMs]
    assert start == max(r[0] for r in ranges)
    assert stop == min(r[1] for r in ranges)
    for s, e in ranges:                     # every shared row is a valid row of every trial
        assert s <= start and stop <= e
    if len(set(dms)) == 1:
        assert (start, stop) == ranges[0]
    assert common_crop_range(z, DMs, rf, nsamp=4096) == (
        max(crop_range(z, d, rf, 4096)[0] for d in DMs),
        min(crop_range(z, d, rf, 4096)[1] for d in DMs))


def test_common_crop_can_be_empty():
    z = _signal(n=2 ** 14)
    # each sweep alone fits the block, but they sit at opposite ends of it
    DMs = [pb.DM(1.2), pb.DM(-1.2)]
    for d in DMs:
        s, e = crop_range(z, d, z.max_freq)
        assert e > s
    start, stop = common_crop_range(z, DMs, z.max_freq)
    assert stop <= start


def test_dm_arguments_are_normalised():
    out = as_dm_list([1.5, pb.DM(-2.0), np.float64(0.0), 3])
    assert all(isinstance(d, pb.DM) for d in out)
    assert [d.dm for d in out] == [1.5, -2.0, 0.0, 3.0]
    assert [d.dm for d in as_dm_list(np.array([4.0, -1.0]))] == [4.0, -1.0]
    assert [d.dm for d in as_dm_list((pb.DM(7.0),))] == [7.0]
    with pytest.raises(ValueError):
        as_dm_list([])
    for bad in (3.0, pb.DM(3.0), "3.0", [[1.0, 2.0]]):
        with pytest.raises(TypeError):
            as_dm_list(bad)


def test_argument_errors_come_before_any_device_work():
    z = _signal()
    with pytest.raises(ValueError):
        pb.dedisperse_trials(z, [1.0, 2.0], detect=False, downsample=4)
    with pytest.raises(TypeError):
        pb.dedisperse_trials(np.zeros((16, 2), np.complex64), [1.0])
    with pytest.raises(ValueError):
        pb.dedisperse_trials(z, [])


def test_dask_input_raises(monkeypatch):
    import fake_dask
    da = fake_dask.install(monkeypatch)
    x = np.zeros((4096, 4, 2), np.complex64)
    z = _signal(data=da.from_array(x, chunks=(4096, 2, 2)))
    with pytest.raises(TypeError, match="dedisperse_detect"):
        pb.dedisperse_trials(z, [1.0, 2.0])
    raw = da.from_array(np.zeros((4096, 4, 2, 2), np.int8), chunks=(4096, 2, 2, 2))
    with pytest.raises(TypeError, match="dedisperse_detect"):
        pb.dedisperse_trials((raw, _signal(n=4096, nchan=4)), [1.0])
