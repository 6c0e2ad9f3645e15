"""Single-pulse search of a DM x time plane (builder-defined; kernels.boxcar_search)."""

from typing import NamedTuple

import numpy as np

from .. import _dask, kernels
from ..core import IntensitySignal
from ..device import DeviceArray

__all__ = ["single_pulse_search", "SinglePulseCandidates"]

#: default boxcar widths: 1, 2, 4, ..., 1024 samples
DEFAULT_WIDTHS = tuple(2 ** k for k in range(11))


class SinglePulseCandidates(NamedTuple):
    """Windows whose best boxcar S/N reaches the threshold, sorted by (trial, column, window)."""
    trial: np.ndarray      # int64 index into the list of trials
    column: np.ndarray     # int64 index of the flattened trailing axes of a trial
    sample: np.ndarray     # int64 start of the boxcar, in samples of the trial
    width: np.ndarray      # int32 boxcar width in samples
    snr: np.ndarray        # float32 S/N
    offset_s: np.ndarray   # float64 sample / sample_rate: seconds after the trial's start_time
    stats: np.ndarray      # float64 (ntrial, *trailing, 2): the (mean, std) used per series


def _stack(datas):
    """One new (ntrial, rows, ...) array from trials that are not slabs of one array."""
    if isinstance(datas[0], DeviceArray):
        import torch
        return DeviceArray(torch.stack([d.tensor for d in datas]))
    return np.stack(datas)


def _plane(datas):
    """The (ntrial, rows, ...) plane of the trials' data: a view when they are consecutive
    C-contiguous slabs of one array (what the trial functions return), else a stacked copy."""
    n, d0 = len(datas), datas[0]
    if isinstance(d0, DeviceArray):
        import torch
        ts = [d.tensor for d in datas]
        step, addr, base = ts[0].numel() * ts[0].element_size(), ts[0].data_ptr(), ts[0]._base
        if all(t.is_contiguous() and t.data_ptr() == addr + k * step and
               (n == 1 or (base is not None and t._base is base)) for k, t in enumerate(ts)):
            return DeviceArray(torch.as_strided(ts[0], (n,) + tuple(ts[0].shape),
                                                (ts[0].numel(),) + tuple(ts[0].stride())))
        return _stack(datas)
    step, addr = d0.nbytes, d0.ctypes.data
    if all(isinstance(d, np.ndarray) and d.flags["C_CONTIGUOUS"] and
           d.ctypes.data == addr + k * step and (n == 1 or (d.base is not None and d.base is d0.base))
           for k, d in enumerate(datas)):
        return np.lib.stride_tricks.as_strided(d0, (n,) + d0.shape, (step,) + d0.strides,
                                               writeable=False)
    return _stack(datas)


def single_pulse_search(trials, /, *, widths=None, window=None, threshold=6.0, stats=None):
    """Search trial time series for single pulses: boxcar S/N at several widths, the best
    (S/N, start, width) of each window of ``window`` starts, and the windows at or above
    ``threshold`` as candidates (builder-defined; :func:`kernels.boxcar_search` gives the full
    windowed output).

    ``trials`` is the list returned by :func:`incoherent_dedispersion_trials` or
    :func:`dedisperse_trials` (``IntensitySignal`` objects of one shape, sample rate and start
    time), or one ``IntensitySignal``.  Each column of each trial (the trailing axes flattened) is
    one series, normalised by its own float64 mean and population std, or by ``stats``
    (``(ntrial, *trailing, 2)`` float64 ``(mean, std)``) when given.  ``widths`` defaults to 1, 2,
    4, ..., 1024 samples and ``window`` to ``max(widths)``.

    The search runs on the GPU: trials that are consecutive slabs of one array (as both trial
    functions return) are passed without a copy, others are stacked once; host data is uploaded
    once.  Candidates are selected on the device, so only they cross the bus.  Returns a
    :class:`SinglePulseCandidates` of numpy arrays sorted by (trial, column, window)."""
    if isinstance(trials, IntensitySignal):
        trials = [trials]
    trials = list(trials)
    if not trials:
        raise ValueError("single_pulse_search needs at least one trial")
    for z in trials:
        if not isinstance(z, IntensitySignal):
            raise TypeError("trials must be IntensitySignal objects")
        if _dask.is_dask(z.data):
            raise TypeError("single_pulse_search takes numpy or DeviceArray data (a dask array: "
                            "compute it first)")
        if np.dtype(z.dtype) != np.float32:
            raise TypeError(f"single_pulse_search needs float32 data, got {z.dtype}")
    z0 = trials[0]
    on_dev = isinstance(z0.data, DeviceArray)
    for z in trials[1:]:
        if isinstance(z.data, DeviceArray) != on_dev:
            raise ValueError("trials must all be on the host or all on the device")
        if tuple(z.shape) != tuple(z0.shape):
            raise ValueError(f"trials differ in shape: {z.shape} and {z0.shape}")
        if z.sample_rate_hz != z0.sample_rate_hz:
            raise ValueError("trials differ in sample rate")
        if (z.start_time is None) != (z0.start_time is None) or (
                z.start_time is not None and not z.start_time.isclose(z0.start_time)):
            raise ValueError("trials differ in start time")
    widths = DEFAULT_WIDTHS if widths is None else tuple(int(w) for w in np.atleast_1d(widths))
    window = max(widths) if window is None else int(window)
    if on_dev and len({z.data.device for z in trials}) > 1:
        raise ValueError("trials must all be on one device")

    plane = _plane([z.data for z in trials])
    if not on_dev:
        plane = DeviceArray.from_numpy(plane, kernels.default_device())
    trailing = tuple(plane.shape[2:])
    if stats is not None and not isinstance(stats, DeviceArray):
        stats = DeviceArray.from_numpy(np.ascontiguousarray(stats, dtype=np.float64), plane.device)
    snr, start, width, st = kernels.boxcar_search(plane, widths, window, stats=stats)
    nser, nwin = snr.shape[0], snr.shape[1]
    ncols = int(np.prod(trailing, dtype=np.int64)) if trailing else 1
    # (trial, column, window) order: nonzero walks the permuted view in row-major order
    s3 = snr.tensor.reshape(nser, nwin, ncols).permute(0, 2, 1)
    idx = (s3 >= float(threshold)).nonzero()
    k, c, j = idx[:, 0], idx[:, 1], idx[:, 2]
    sel_snr = s3[k, c, j].cpu().numpy()
    sel_start = start.tensor.reshape(nser, nwin, ncols)[k, j, c].cpu().numpy().astype(np.int64)
    sel_width = width.tensor.reshape(nser, nwin, ncols)[k, j, c].cpu().numpy()
    idx = idx.cpu().numpy()
    return SinglePulseCandidates(trial=idx[:, 0].astype(np.int64),
                                 column=idx[:, 1].astype(np.int64), sample=sel_start,
                                 width=sel_width, snr=sel_snr,
                                 offset_s=sel_start / float(z0.sample_rate_hz),
                                 stats=st.numpy())
