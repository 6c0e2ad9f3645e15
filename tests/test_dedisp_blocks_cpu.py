"""Host logic of pb.overlap_save_dedispersion: its block schedule (shared with pb.dedisperse_fold)
and the validation of its arguments, which happens before any device work.  No GPU needed."""

import numpy as np
import pytest

import pulsarbat_b200 as pb
from pulsarbat_b200.transforms import dedispersion

SR, FCEN = 6.25e6, 625e6


def _signal(n=2 ** 14, nchan=8, data=None):
    x = np.zeros((n, nchan, 2), np.complex64) if data is None else data
    return pb.DualPolarizationSignal(x, sample_rate=SR * pb.units.Hz,
                                     center_freq=FCEN * pb.units.Hz, pol_type="linear")


def test_block_schedule_lives_with_overlap_save_and_folding_shares_it():
    from pulsarbat_b200.pulsar import folding
    assert folding._block_schedule is dedispersion._block_schedule
    assert dedispersion._block_schedule.__module__ == dedispersion.__name__


@pytest.mark.parametrize("nsamp, ds", [(10 * 4096, 1), (10 * 4096, 8), (4096, 1), (4095, 1)])
def test_block_schedule_of_a_stream(nsamp, ds):
    z = _signal(n=nsamp)
    start, stop = dedispersion.crop_range(z, pb.DM(0.05), z.center_freq, nsamp=4096)
    advance, starts = dedispersion._block_schedule(nsamp, 4096, start, stop, ds)
    assert advance % ds == 0 and stop - start - ds < advance <= stop - start
    assert starts == [b * advance for b in range(len(starts))]
    assert (len(starts) - 1) * advance + 4096 <= nsamp if starts else nsamp < 4096
    assert starts == [] or starts[-1] + advance + 4096 > nsamp     # the tail does not fill a block


def test_argument_errors_come_before_any_device_work():
    z = _signal()
    dm = pb.DM(0.05)                          # a sweep of about 500 of 4096 samples
    with pytest.raises(ValueError, match="downsample"):
        pb.overlap_save_dedispersion(z, dm, 4096, detect=True, downsample=0)
    with pytest.raises(ValueError, match="detect=True"):
        pb.overlap_save_dedispersion(z, dm, 4096, downsample=4)
    with pytest.raises(ValueError, match="detect=True"):
        pb.overlap_save_dedispersion(z, dm, 4096, stokes_I=True)
    with pytest.raises(TypeError):
        pb.overlap_save_dedispersion(np.zeros((4096, 2), np.complex64), dm, 4096)
    with pytest.raises(TypeError):
        pb.overlap_save_dedispersion((np.zeros((4096, 8, 2, 2), np.int8), None), dm, 4096)
    with pytest.raises(ValueError, match="sweep"):
        pb.overlap_save_dedispersion(z, pb.DM(0.5), 4096)
    with pytest.raises(ValueError, match="shorter than downsample"):
        pb.overlap_save_dedispersion(z, dm, 4096, detect=True, downsample=4096)


def test_kernel_call_takes_device_streams_only():
    with pytest.raises(TypeError, match="DeviceArray"):
        pb.kernels.dedisperse_overlap_save(
            np.zeros((4096, 8, 2), np.complex64), block_len=1024, dm=0.5, sample_rate_hz=SR,
            chan_freq_hz=np.full(8, FCEN), ref_freq_hz=FCEN, crop=(10, 1000))
