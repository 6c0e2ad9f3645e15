"""Dedispersion: GPU-backed mirror of the reference's ``transforms/dedispersion.py``.

``coherent_dedispersion`` keeps the reference signature, return type, metadata update and
exceptions (dedispersion.py:81-133); the FFT, the chirp and the inverse FFT run as fused
sm_100a passes in libpbk (the chirp is generated in registers and never stored).
"""

import math

import numpy as np

from .. import _dask
from .. import _lib as L
from .. import kernels
from .. import units as u
from ..core import BasebandSignal, IntensitySignal, RadioSignal

__all__ = ["DispersionMeasure", "DM", "coherent_dedispersion", "incoherent_dedispersion",
           "dedisperse_detect", "dedisperse_trials", "incoherent_dedispersion_trials",
           "overlap_save_dedispersion"]

#: s MHz^2 cm^3 / pc -- dedispersion.py:30
DISPERSION_CONSTANT = 1.0 / 2.41e-4


def _hz(q):
    """Frequency in Hz; bare infinities are allowed as reference frequencies
    (reference tests/test_dedispersion.py:16-19 pass ``np.inf``)."""
    if isinstance(q, (int, float, np.floating)) and math.isinf(q):
        return float(q)
    return float(u.to_value(q, u.Hz))


class DispersionMeasure(u.Quantity):
    """Dispersion measure in pc / cm^3 (dedispersion.py:26-75)."""

    dispersion_constant = DISPERSION_CONSTANT

    def __init__(self, value, unit=None):
        if isinstance(value, u.Quantity):
            value = value.to_value(u.dm_unit)
        elif hasattr(value, "to_value"):
            value = float(value.to_value("pc / cm3"))
        super().__init__(value, u.dm_unit)

    def __neg__(self):
        return DispersionMeasure(-self.value)

    def __mul__(self, other):
        r = super().__mul__(other)
        return DispersionMeasure(r.value) if r.unit == u.dm_unit else r

    __rmul__ = __mul__

    @property
    def dm(self):
        return float(self.value)

    def time_delay(self, f, ref_freq):
        """Delay of frequency ``f`` relative to ``ref_freq`` (dedispersion.py:32-36)."""
        f_mhz = np.asarray(_hz_array(f)) / 1e6
        r_mhz = _hz(ref_freq) / 1e6
        with np.errstate(divide="ignore"):
            delay = self.dispersion_constant * self.value * (1 / f_mhz ** 2 - 1 / r_mhz ** 2)
        return u.Quantity(delay, u.s)

    def sample_delay(self, f, ref_freq, sample_rate):
        """Delay in (fractional) samples (dedispersion.py:38-42)."""
        d = self.time_delay(f, ref_freq).to_value(u.s) * float(u.to_value(sample_rate, u.Hz))
        return float(d) if np.ndim(d) == 0 else d

    def chirp_function(self, N, dt, center_freq, ref_freq):
        """(N,) complex64 transfer function for one channel (dedispersion.py:44-57)."""
        sr = 1.0 / float(u.to_value(dt, u.s))
        return kernels.chirp(int(N), 1, dm=self.dm, sample_rate_hz=sr,
                             ref_freq_hz=_hz(ref_freq), chan_freq_hz=[_hz(center_freq)])[:, 0]

    def chirp_from_signal(self, z, /, *, ref_freq=None):
        """(N, nchan, 1, ...) complex64 chirp for ``z`` (dedispersion.py:59-75)."""
        if not isinstance(z, BasebandSignal):
            raise TypeError("Signal must be a BasebandSignal object.")
        if ref_freq is None:
            ref_freq = z.center_freq
        c = kernels.chirp(len(z), z.nchan, dm=self.dm, sample_rate_hz=z.sample_rate_hz,
                          ref_freq_hz=_hz(ref_freq), chan_freq_hz=z.channel_freqs_hz)
        return c.reshape(c.shape + (1,) * (z.ndim - 2))


DM = DispersionMeasure


def _hz_array(f):
    if isinstance(f, (int, float, np.floating, np.ndarray)) and np.all(np.isinf(f)):
        return np.asarray(f, dtype=float)
    return np.asarray(u.to_value(f, u.Hz), dtype=float)


def _as_dm(x):
    return x if isinstance(x, DispersionMeasure) else DispersionMeasure(x)


def crop_range(z, dm, ref_freq, nsamp=None):
    """(start, stop) exactly as dedispersion.py:127-131, for a block of ``nsamp`` samples of ``z``
    (default: all of it)."""
    d_top = dm.sample_delay(z.max_freq, ref_freq, z.sample_rate)
    d_bot = dm.sample_delay(z.min_freq, ref_freq, z.sample_rate)
    start = math.ceil(-min(0, d_top, d_bot))
    stop = (len(z) if nsamp is None else nsamp) - math.ceil(+max(0, d_top, d_bot))
    return start, stop


def _cropped_like(cls, z, data, start, **kw):
    """``cls.like(z, x)[start:stop]`` for data that is already cropped: same start_time update as
    core.py:162-163."""
    if z.start_time is not None:
        kw.setdefault("start_time", z.start_time + start / z.sample_rate)
    return cls.like(z, data, **kw)


def coherent_dedispersion(z, DM, /, *, ref_freq=None, chirp=None):
    """Coherently dedisperse a baseband signal (drop-in for dedispersion.py:81-133).

    Returns ``type(z)`` cropped at both ends by the dispersion sweep; raises ``TypeError`` for
    non-baseband input.  With ``chirp=`` the given array multiplies the spectrum instead of the
    generated chirp (dedispersion.py:121-124).  Any length works (powers of two are the fast
    path); there is no CPU fallback.
    """
    if not isinstance(z, BasebandSignal):
        raise TypeError("Signal must be a BasebandSignal object.")
    DM = _as_dm(DM)
    if ref_freq is None:
        ref_freq = z.center_freq
    start, stop = crop_range(z, DM, ref_freq)
    if _dask.is_dask(z.data):
        # lazy input: one GPU call per channel chunk when the result is computed, every chunk
        # with ITS channel frequencies and the GLOBAL ref_freq and crop (transforms.py:49-50)
        freqs, sr, rf, dm = z.channel_freqs_hz, z.sample_rate_hz, _hz(ref_freq), DM.dm
        ch = None if chirp is None else np.asarray(chirp).reshape(len(z), z.nchan)

        def chunk(block, lo, hi):
            return np.asarray(kernels.dedisperse(
                np.asarray(block), dm=dm, sample_rate_hz=sr, chan_freq_hz=freqs[lo:hi],
                ref_freq_hz=rf, crop=(start, stop),
                chirp_array=None if ch is None else ch[:, lo:hi]))
        x = _dask.map_channel_chunks(z.data, chunk, out_rows=max(0, stop - start),
                                     out_dtype=z.dtype)
    else:
        x = kernels.dedisperse(z.data, dm=DM.dm, sample_rate_hz=z.sample_rate_hz,
                               chan_freq_hz=z.channel_freqs_hz, ref_freq_hz=_hz(ref_freq),
                               crop=(start, stop), chirp_array=chirp)
    if stop <= start:
        # empty crop: the reference would hand back a zero-length slice (dedispersion.py:133)
        start = min(start, len(z))
    return _cropped_like(type(z), z, x, start)


def incoherent_delays(z, DM, ref_freq):
    """(delays, N_out, crop_before) exactly as dedispersion.py:164-169."""
    delays = np.asarray(DM.sample_delay(z.channel_freqs, ref_freq, z.sample_rate), dtype=float)
    delays = np.atleast_1d(delays).round().astype(np.int64)
    crop_before = -min(0, int(delays[0]), int(delays[-1]))
    delays = delays + crop_before
    return delays, len(z) - int(max(delays)), crop_before


def incoherent_dedispersion(z, DM, /, *, ref_freq=None):
    """Incoherently dedisperse a signal: per-channel integer roll and crop (drop-in for
    dedispersion.py:136-177; same TypeError, crop and start_time update).  Any real or complex
    RadioSignal; the roll is a bit-exact gather on the GPU."""
    if not isinstance(z, RadioSignal):
        raise TypeError("Signal must be a RadioSignal object.")
    DM = _as_dm(DM)
    if ref_freq is None:
        ref_freq = z.center_freq
    delays, n_out, crop_before = incoherent_delays(z, DM, ref_freq)
    if n_out < 0 or int(delays.min()) < 0:
        # numpy's negative slices would wrap here (sweep longer than the signal); refuse instead
        raise ValueError("dispersion sweep exceeds the signal length")
    x = kernels.shift_channels(z.data, delays, n_out)
    kw = {}
    if crop_before and z.start_time is not None:
        kw["start_time"] = z.start_time + crop_before / z.sample_rate
    return type(z).like(z, x, **kw)


def dedisperse_detect(z, DM, /, *, ref_freq=None, stokes_I=False, downsample=1, crop=True):
    """Fused coherent dedispersion -> power detection -> time sum in one plan.

    Equivalent to ``coherent_dedispersion(z, DM).to_intensity()`` (or ``to_stokes_I``) followed by
    summing ``downsample`` consecutive samples, without materialising the dedispersed voltages.
    ``crop=False`` keeps the whole circular result (for configurations whose sweep exceeds the
    block, SURVEY.md 0.5).  Accepts int8 (re, im) pairs in a trailing axis of length 2 when
    ``z`` is given as a tuple ``(raw_int8, template_signal)``.
    """
    raw = None
    if isinstance(z, tuple):
        raw, z = z
    if not isinstance(z, BasebandSignal):
        raise TypeError("Signal must be a BasebandSignal object.")
    DM = _as_dm(DM)
    if ref_freq is None:
        ref_freq = z.center_freq
    start, stop = crop_range(z, DM, ref_freq) if crop else (0, len(z))
    kind = L.OUT_STOKES_I if stokes_I else L.OUT_INTENSITY
    src = z.data if raw is None else raw
    if _dask.is_dask(src):
        freqs, sr, rf, dm = z.channel_freqs_hz, z.sample_rate_hz, _hz(ref_freq), DM.dm

        def chunk(block, lo, hi):
            return np.asarray(kernels.dedisperse(
                np.asarray(block), dm=dm, sample_rate_hz=sr, chan_freq_hz=freqs[lo:hi],
                ref_freq_hz=rf, crop=(start, stop), out_kind=kind, downsample=downsample,
                int8=raw is not None))
        rows = max(0, stop - start) // int(downsample)
        if raw is not None:        # (N, C, P, 2) int8: the (re, im) axis never survives
            def chunk_raw(block, lo, hi):
                y = chunk(block, lo, hi)
                return y.reshape(y.shape + (1,) * (block.ndim - y.ndim))
            x = _dask.map_channel_chunks(src, chunk_raw, out_rows=rows, out_dtype=np.float32)
            x = x.reshape(x.shape[:2] + (() if stokes_I else tuple(z.shape[2:])))
        else:
            x = _dask.map_channel_chunks(src, chunk, out_rows=rows, drop_trailing=stokes_I,
                                         out_dtype=_dask.real_dtype_of(z.dtype))
    else:
        x = kernels.dedisperse(src, dm=DM.dm, sample_rate_hz=z.sample_rate_hz,
                               chan_freq_hz=z.channel_freqs_hz, ref_freq_hz=_hz(ref_freq),
                               crop=(start, stop), out_kind=kind, downsample=downsample,
                               int8=raw is not None)
    kw = {"chan_bw": z.chan_bw}
    if downsample > 1:
        kw["sample_rate"] = z.sample_rate / downsample
    return _cropped_like(IntensitySignal, z, x, max(start, 0), **kw)


def as_dm_list(DMs):
    """A sequence of DM values or DispersionMeasures as a list of DispersionMeasures."""
    if isinstance(DMs, (str, bytes)) or np.ndim(DMs) != 1:
        raise TypeError("DMs must be a one-dimensional sequence of dispersion measures")
    out = [_as_dm(d) for d in DMs]
    if not out:
        raise ValueError("DMs must hold at least one dispersion measure")
    return out


def common_crop_range(z, DMs, ref_freq, nsamp=None):
    """(start, stop) valid for every DM of ``DMs``: the intersection of their :func:`crop_range`,
    i.e. the latest start and the earliest stop.  ``stop <= start`` when it is empty."""
    ranges = [crop_range(z, dm, ref_freq, nsamp) for dm in DMs]
    return max(r[0] for r in ranges), min(r[1] for r in ranges)


def dedisperse_trials(z, DMs, /, *, ref_freq=None, detect=True, stokes_I=False, downsample=1,
                      crop=True):
    """Coherently dedisperse one block at several trial DMs (a DM search, or refining the DM of a
    known pulsar), sharing the forward FFT of the block between the trials.

    Returns a list with one signal per DM: ``IntensitySignal`` objects (per-pol power, or Stokes I
    with ``stokes_I=True``, summed over ``downsample`` samples), or ``type(z)`` voltages with
    ``detect=False``.  Their data are views of one stacked array.  With ``crop=True`` all trials
    share one crop, the intersection of every DM's crop (:func:`common_crop_range`), so every row
    is valid for every trial and all results have the same ``start_time`` and length; element k
    then equals ``dedisperse_detect(z, DMs[k])`` cut to that crop.  An empty intersection gives
    zero-row results.  ``z`` may be a ``(raw_int8, template_signal)`` tuple as in
    :func:`dedisperse_detect`.  Dask input raises ``TypeError``.
    """
    raw = None
    if isinstance(z, tuple):
        raw, z = z
    if not isinstance(z, BasebandSignal):
        raise TypeError("Signal must be a BasebandSignal object.")
    DMs = as_dm_list(DMs)
    if not detect and (downsample > 1 or stokes_I):
        raise ValueError("downsample and stokes_I need detect=True")
    src = z.data if raw is None else raw
    if _dask.is_dask(src):
        raise TypeError("dedisperse_trials takes numpy or DeviceArray blocks (a dask array: "
                        "compute the block first, or call dedisperse_detect per chunk)")
    if ref_freq is None:
        ref_freq = z.center_freq
    start, stop = common_crop_range(z, DMs, ref_freq) if crop else (0, len(z))
    kind = (L.OUT_C64 if not detect else L.OUT_STOKES_I if stokes_I else L.OUT_INTENSITY)
    x = kernels.dedisperse_trials(src, dms=[d.dm for d in DMs], sample_rate_hz=z.sample_rate_hz,
                                  chan_freq_hz=z.channel_freqs_hz, ref_freq_hz=_hz(ref_freq),
                                  crop=(start, stop), out_kind=kind, downsample=downsample,
                                  raw=None if raw is None else "int8")
    if not detect:
        start = min(start, len(z)) if stop <= start else start
        return [_cropped_like(type(z), z, x[k], start) for k in range(len(DMs))]
    kw = {"chan_bw": z.chan_bw}
    if downsample > 1:
        kw["sample_rate"] = z.sample_rate / downsample
    return [_cropped_like(IntensitySignal, z, x[k], max(start, 0), **kw) for k in range(len(DMs))]


def incoherent_trial_delays(z, DMs, ref_freq):
    """``(e, t_lo, rows)`` of :func:`incoherent_dedispersion_trials`: trial k reads input row
    ``t_lo + j + r_k[c]`` of channel c for its output row j, where ``r_k`` are the reference's
    rounded delays (:func:`incoherent_delays` without its ``crop_before`` shift) and
    ``[t_lo, t_lo + rows)`` is the intersection of every trial's valid rows in absolute input rows.
    ``e`` is the (ndm, nchan) int64 table ``r_k[c] + t_lo``; ``rows`` is 0 when the intersection
    is empty.  A DM whose sweep exceeds the signal raises ``ValueError``."""
    tables, lo, hi = [], [], []
    for dm in as_dm_list(DMs):
        delays, n_out, crop_before = incoherent_delays(z, dm, ref_freq)
        if n_out < 0 or int(delays.min()) < 0:
            raise ValueError("dispersion sweep exceeds the signal length")
        tables.append(delays - crop_before)
        lo.append(crop_before)
        hi.append(crop_before + n_out)
    t_lo = max(lo)
    rows = max(0, min(hi) - t_lo)
    return np.stack(tables) + t_lo, t_lo, rows


def incoherent_dedispersion_trials(z, DMs, /, *, ref_freq=None):
    """Incoherently dedisperse a filterbank at several trial DMs and sum over frequency: a DM x
    time plane in one GPU call (builder-defined; kernels.incoherent_trials).

    Returns a list with one ``IntensitySignal`` per DM, each of shape ``(rows, 1, ...)``, views
    of one stacked array on ``z``'s side of the bus.  Element k equals
    ``incoherent_dedispersion(z, DMs[k]).data`` summed over the frequency axis (in float32,
    channels in ascending order) and cut to the rows that are valid for every trial
    (:func:`incoherent_trial_delays`); an empty intersection gives zero-row results.  Each result
    keeps the sample rate and the band (one channel of ``chan_bw * nchan`` at ``center_freq``,
    ``freq_align="center"``) and starts ``t_lo`` samples after ``z``.  ``z`` must hold float32
    data (a filterbank, ``stft_detect`` or ``dedisperse_detect`` output); other dtypes and dask
    arrays raise ``TypeError``.
    """
    if not isinstance(z, RadioSignal):
        raise TypeError("Signal must be a RadioSignal object.")
    if _dask.is_dask(z.data):
        raise TypeError("incoherent_dedispersion_trials takes numpy or DeviceArray data (a dask "
                        "array: compute it first, or call incoherent_dedispersion per chunk)")
    if np.dtype(z.dtype) != np.float32:
        raise TypeError(f"incoherent_dedispersion_trials needs float32 data, got {z.dtype} "
                        "(complex and float64 signals are not supported)")
    DMs = as_dm_list(DMs)
    if ref_freq is None:
        ref_freq = z.center_freq
    e, t_lo, rows = incoherent_trial_delays(z, DMs, ref_freq)
    trailing = tuple(z.shape[2:])
    if rows:
        x = kernels.incoherent_trials(z.data, e, rows)
    elif isinstance(z.data, kernels.DeviceArray):
        x = kernels.DeviceArray.empty((len(DMs), 0) + trailing, np.float32, z.data.device)
    else:
        x = np.empty((len(DMs), 0) + trailing, np.float32)
    shape = (len(DMs), rows, 1) + trailing
    if isinstance(x, kernels.DeviceArray):
        x = kernels.DeviceArray(x.tensor.reshape(shape))
    else:
        x = x.reshape(shape)
    kw = {"chan_bw": z.chan_bw * z.nchan, "center_freq": z.center_freq, "freq_align": "center"}
    if z.start_time is not None:
        kw["start_time"] = z.start_time + t_lo / z.sample_rate
    return [IntensitySignal.like(z, x[k], **kw) for k in range(len(DMs))]


def _block_schedule(nsamp, block_len, start, stop, downsample):
    """Overlap-save blocks of a stream: ``(advance, block starts)``.  Blocks of ``block_len``
    samples keep the rows ``[start, start + advance)``, where the advance is the valid length
    ``stop - start`` rounded down to a multiple of ``downsample`` (every summed output row lies
    inside one block); a tail that does not fill a block is dropped."""
    valid = stop - start
    if valid <= 0:
        raise ValueError("block length does not exceed the dispersion sweep")
    advance = valid // downsample * downsample
    if advance == 0:
        raise ValueError(f"the valid length of a block ({valid} samples) is shorter than "
                         f"downsample={downsample}")
    return advance, list(range(0, nsamp - block_len + 1, advance))


def overlap_save_dedispersion(z, DM, block_len, /, *, ref_freq=None, detect=False, stokes_I=False,
                              downsample=1):
    """Dedisperse a long stream in overlapping blocks of ``block_len`` samples (builder-defined,
    SURVEY.md 8a row O).  The blocks advance by the valid length of a block rounded down to a
    multiple of ``downsample`` and keep that many rows after the leading crop; the tail that does
    not fill a block is dropped.

    With ``detect=False`` the result equals the concatenation of ``coherent_dedispersion`` applied
    to those blocks, i.e. what the reference gives per block.  With ``detect=True`` it is an
    ``IntensitySignal``: the concatenation of ``dedisperse_detect(block, DM, stokes_I=...,
    downsample=...)`` over the blocks, which is what ``dedisperse_fold(..., block_len=...)`` folds.
    ``z`` may be a ``(raw_int8, template_signal)`` tuple as in :func:`dedisperse_detect`.

    A stream on the device (a ``DeviceArray``, complex64 or raw) is dedispersed by one library
    call for all blocks (:func:`kernels.dedisperse_overlap_save`) and the result stays on the
    device.  Host complex64 and int8 streams go through the three-stream pipeline (upload, kernels
    and download of consecutive blocks overlap); complex128 runs the FP64 kernels per block.
    """
    raw = None
    if isinstance(z, tuple):
        raw, z = z
    if not isinstance(z, BasebandSignal):
        raise TypeError("Signal must be a BasebandSignal object.")
    ds = int(downsample)
    if ds < 1:
        raise ValueError("downsample must be >= 1")
    if not detect and (ds > 1 or stokes_I):
        raise ValueError("downsample and stokes_I need detect=True")
    DM = _as_dm(DM)
    if ref_freq is None:
        ref_freq = z.center_freq
    block_len = int(block_len)
    src = z.data if raw is None else raw
    start, stop = crop_range(z, DM, ref_freq, nsamp=block_len)
    advance, starts = _block_schedule(src.shape[0], block_len, start, stop, ds)
    kind = (L.OUT_C64 if not detect else L.OUT_STOKES_I if stokes_I else L.OUT_INTENSITY)
    kw = dict(dm=DM.dm, sample_rate_hz=z.sample_rate_hz, chan_freq_hz=z.channel_freqs_hz,
              ref_freq_hz=_hz(ref_freq), crop=(start, start + advance), out_kind=kind,
              downsample=ds, raw=None if raw is None else "int8")
    on_dev = isinstance(src, kernels.DeviceArray)
    if on_dev and (raw is not None or src.dtype == np.complex64):
        data = kernels.dedisperse_overlap_save(src, block_len=block_len, **kw)
    elif raw is None and (on_dev or np.asarray(src).dtype != np.complex64):
        # complex128: the FP64 kernels block by block, on the stream's side of the bus
        pieces = [kernels.dedisperse(src[b:b + block_len], **kw) for b in starts]
        if not pieces:
            shape = (0,) + (tuple(z.shape[1:]) if kind != L.OUT_STOKES_I else (z.nchan,))
            dt = np.complex128 if kind == L.OUT_C64 else np.float64
            data = kernels.DeviceArray.empty(shape, dt, src.device) if on_dev else np.empty(shape, dt)
        elif on_dev:
            import torch
            data = kernels.DeviceArray(torch.cat([p.tensor for p in pieces]))
        else:
            data = np.concatenate(pieces, axis=0)
    else:
        # host complex64 or int8 stream: the blocks go through the three-stream pipeline (upload of
        # block i+1, kernels of block i and download of block i-1 overlap) straight into the result
        from .. import streaming
        src = np.asarray(src)
        rows = advance // ds
        trailing = (z.nchan,) if kind == L.OUT_STOKES_I else tuple(z.shape[1:])
        data = np.empty((len(starts) * rows,) + trailing,
                        np.complex64 if kind == L.OUT_C64 else np.float32)
        blocks = (src[b:b + block_len] for b in starts)
        for i, y in enumerate(streaming.dedisperse_blocks(blocks, pinned_out=True, **kw)):
            data[i * rows:(i + 1) * rows] = y
    if not detect:
        return _cropped_like(type(z), z, data, start)
    kw = {"chan_bw": z.chan_bw}
    if ds > 1:
        kw["sample_rate"] = z.sample_rate / ds
    return _cropped_like(IntensitySignal, z, data, start, **kw)
